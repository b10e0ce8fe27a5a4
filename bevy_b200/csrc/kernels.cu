// kernels.cu -- the sm_100a kernels of libb200vis: propagate -> cull -> cluster.
//
// Numerics contract: every float operation below is IEEE-754 binary32 in the
// operation order of glam's x86-64/SSE2 backend (SURVEY.md Appendix A), with
// NO fused multiply-add (this translation unit is compiled with -fmad=false,
// -prec-div=true, -prec-sqrt=true, -ftz=false), so the float compares that
// decide ViewVisibility bits and cluster membership are bit-identical to the
// reference's CPU systems.  These are HBM-bound byte/float streaming kernels:
// no tensor cores on purpose (SURVEY.md 8d: ~1.3 flop/B).
#include <cstdint>
#include <cstdlib>
#include <cuda_runtime.h>

#include "device_types.cuh"
#include "kernels.cuh"

namespace b200vis {

// ------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------
struct Aff { float4 r0, r1, r2; };   // row form of a glam Affine3A: rK = (X[k], Y[k], Z[k], T[k])

// Transform::compute_affine = Affine3A::from_scale_rotation_translation
// (crates/bevy_transform/src/components/transform.rs:273-275; glam Mat3A::from_quat)
__device__ __forceinline__ Aff affine_from_trs(float4 A, float4 q, float2 C) {
    const float sx = A.w, sy = C.x, sz = C.y;
    const float x2 = q.x + q.x, y2 = q.y + q.y, z2 = q.z + q.z;
    const float xx = q.x * x2, xy = q.x * y2, xz = q.x * z2;
    const float yy = q.y * y2, yz = q.y * z2, zz = q.z * z2;
    const float wx = q.w * x2, wy = q.w * y2, wz = q.w * z2;
    Aff a;
    a.r0 = make_float4((1.0f - (yy + zz)) * sx, (xy - wz) * sy, (xz + wy) * sz, A.x);
    a.r1 = make_float4((xy + wz) * sx, (1.0f - (xx + zz)) * sy, (yz - wx) * sz, A.y);
    a.r2 = make_float4((xz - wy) * sx, (yz + wx) * sy, (1.0f - (xx + yy)) * sz, A.z);
    return a;
}

// one output row of Affine3A * Affine3A (global_transform.rs:315-317):
//   matrix3 = P.m3 * L.m3 with mul_vec3a = ((X*v.x) + (Y*v.y)) + (Z*v.z); translation = P.m3*L.t + P.t
__device__ __forceinline__ float4 affine_mul_row(float4 p, const Aff &l) {
    float4 r;
    r.x = (p.x * l.r0.x + p.y * l.r1.x) + p.z * l.r2.x;
    r.y = (p.x * l.r0.y + p.y * l.r1.y) + p.z * l.r2.y;
    r.z = (p.x * l.r0.z + p.y * l.r1.z) + p.z * l.r2.z;
    r.w = ((p.x * l.r0.w + p.y * l.r1.w) + p.z * l.r2.w) + p.w;
    return r;
}
__device__ __forceinline__ bool row_neq(float4 a, float4 b) {
    return (a.x != b.x) | (a.y != b.y) | (a.z != b.z) | (a.w != b.w);
}
// glam SSE2 dot4 of a plane with (p, 1): (n.x*p.x + n.z*p.z) + (n.y*p.y + n.w*1)
__device__ __forceinline__ float plane_dot_point(float4 n, float px, float py, float pz) {
    return (n.x * px + n.z * pz) + (n.y * py + n.w * 1.0f);
}
__device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz) {
    return (ax * bx + ay * by) + az * bz;
}
// RenderLayers::intersects (render_layers.rs:121-135): any block-wise AND over the common prefix; block 0 is `elayers`
__device__ __forceinline__ bool layers_intersect(const Rows &R, const CullViews &cvw, uint32_t row, uint32_t v, unsigned long long elayers) {
    if (cvw.layers[v] & elayers) return true;
    if (R.layers_ext == nullptr) return false;
    const uint64_t *e = R.layers_ext + (size_t)row * 3;
    return ((cvw.layers_ext[v][0] & e[0]) | (cvw.layers_ext[v][1] & e[1]) | (cvw.layers_ext[v][2] & e[2])) != 0ull;
}
__device__ __forceinline__ float gl_min(float a, float b) { return a < b ? a : b; }   // glam / SSE min,max
__device__ __forceinline__ float gl_max(float a, float b) { return a > b ? a : b; }

// ------------------------------------------------------------------------------------------
// Warp-level view rejection.  Thirty-two consecutive rows are neighbours in space (one level of one tree, a stretch of a
// spiral of cubes), and a view's frustum holds a small part of the world: before the per-row plane tests of a view, the warp
// builds an axis-aligned box around its rows' bounding-sphere centres (+ the largest radius) and lets 5 x n_views lanes test
// one (view, plane) pair each against it.  A plane the whole box is behind -- by more than the float error any of the exact
// evaluations can carry -- culls every row in Frustum::intersects_sphere already (primitives.rs:255-268), so the view's
// ~70 instructions per row are skipped and every row simply reports "not visible" for it: same bits, less work.
// Rows that are not frustum-tested (no bounds, NoFrustumCulling) or carry non-finite numbers switch the shortcut off for
// their warp.  Returns a bit per view.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int float_order(float f) { const int b = __float_as_int(f); return b ^ ((b >> 31) & 0x7FFFFFFF); }
__device__ __forceinline__ float order_float(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7FFFFFFF)); }
__device__ __forceinline__ uint32_t warp_view_reject(const CullViews &cvw, bool testable, bool blocks, float cx, float cy, float cz, float radius) {
    const float inf = __int_as_float(0x7f800000);
    const bool fin = testable && isfinite(((cx + cy) + cz) + radius);
    if (__any_sync(0xFFFFFFFFu, blocks || (testable && !fin))) return 0u;
    const float x0 = order_float(__reduce_min_sync(0xFFFFFFFFu, float_order(fin ? cx : inf)));
    const float y0 = order_float(__reduce_min_sync(0xFFFFFFFFu, float_order(fin ? cy : inf)));
    const float z0 = order_float(__reduce_min_sync(0xFFFFFFFFu, float_order(fin ? cz : inf)));
    const float x1 = order_float(__reduce_max_sync(0xFFFFFFFFu, float_order(fin ? cx : -inf)));
    const float y1 = order_float(__reduce_max_sync(0xFFFFFFFFu, float_order(fin ? cy : -inf)));
    const float z1 = order_float(__reduce_max_sync(0xFFFFFFFFu, float_order(fin ? cz : -inf)));
    const float r1 = order_float(__reduce_max_sync(0xFFFFFFFFu, float_order(fin ? radius : -inf)));
    if (!(x0 <= x1)) return 0xFFFFFFFFu;          // no frustum-tested row in this warp (and none that blocks): nothing can be visible
    const uint32_t lane = threadIdx.x & 31u;
    bool rej = false;
    if (lane < 5u * cvw.n_views && lane < 30u) {       // views 0..5; a seventh or eighth view is never rejected here
        const float4 n = cvw.planes[lane / 5u][lane % 5u];
        const float m = ((fmaxf(n.x * x0, n.x * x1) + fmaxf(n.y * y0, n.y * y1)) + fmaxf(n.z * z0, n.z * z1)) + n.w;
        const float mag = ((fabsf(n.x) * fmaxf(fabsf(x0), fabsf(x1)) + fabsf(n.y) * fmaxf(fabsf(y0), fabsf(y1))) +
                           fabsf(n.z) * fmaxf(fabsf(z0), fabsf(z1))) + (fabsf(n.w) + fabsf(r1));
        rej = (m + r1) + (1e-5f * mag + 1e-6f) < 0.0f;     // ~25x the rounding any exact plane_dot_point(..) + radius can carry
    }
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, rej);
    uint32_t out = 0;
#pragma unroll
    for (uint32_t v = 0; v < 6u; ++v) out |= ((b >> (5u * v)) & 0x1Fu) ? (1u << v) : 0u;
    return out;
}

// ------------------------------------------------------------------------------------------
// Kernel 1: fused propagate -> cull over one tile of rows per CTA.
//
// A tile is a contiguous row range whose hierarchy edges stay inside the tile (parents in
// shared memory) or point at rows finished by an earlier pass (parents read from HBM).
//   phase 1  all rows: coalesced float4 loads of Transform, old GlobalTransform, bounds, flags
//            (everything a row needs is requested up front: ~11 independent loads per thread)
//   phase 2  per in-tile depth level: GT = parentGT * local, parent matrices staged in shared
//            memory; a level whose parents all sit in the same warp only needs __syncwarp
//            (the planner marks those levels), the others a CTA barrier
//   phase 3  all rows: set_if_neq write-back, frustum tests for every view (branch-free sphere
//            pre-test, OBB test for the survivors), warp-ballot bits into the rank-ordered
//            visible mask, ViewVisibility state machine, change flags
// Template flags: PROP / CULL = stages fused into this launch; SIMPLE = no per-row RenderLayers /
// VisibleEntityRanges / rank columns (every entity on the default layer, rows already in
// Entity::to_bits() order), which removes three loads and the per-lane atomics.
// ------------------------------------------------------------------------------------------
struct TileSmem {
    float4 g0[kTileRows], g1[kTileRows], g2[kTileRows];
    uint16_t parent[kTileRows];
    uint8_t st[kTileRows];       // bit0 visited, bit1 gt changed
    uint8_t dirty[kTileRows];    // TransformTreeChanged this frame (mark_dirty_trees)
};

// VisibleEntityRanges bits of one row: the uploaded column, or -- when the VisibilityRange columns are resident
// (SURVEY 8(f) N4) -- check_visibility_ranges itself (crates/bevy_camera/src/visibility/range.rs:230-284) on this
// frame's GlobalTransform, stored so that the shim can rebuild the resource from it.
__device__ __forceinline__ uint32_t range_mask_of(const Rows &R, uint32_t row, bool has_aabb, float cx, float cy, float cz, const Aff &g) {
    if (R.range_se == nullptr) return R.range[row];
    const float2 se = R.range_se[row];
    // (use_aabb, Some(aabb)) => transform_point3a(aabb.center) -- the cull phase's centre; otherwise the translation
    const bool centre = has_aabb && R.range_use_aabb[row];
    const float mx = centre ? cx : g.r0.w, my = centre ? cy : g.r1.w, mz = centre ? cz : g.r2.w;
    uint32_t m = 0;
    for (uint32_t v = 0; v < R.n_range_views; ++v) {
        const float4 p = R.range_views[v];
        const float dx = p.x - mx, dy = p.y - my, dz = p.z - mz;
        const float d = sqrtf((dx * dx + dy * dy) + dz * dz);            // Vec3A::length
        if (d >= se.x && d < se.y) m |= 1u << v;                         // is_visible_at_all (range.rs:157-159)
    }
    R.range[row] = m;
    return m;
}

template <bool PROP, bool CULL, bool SIMPLE>
__global__ void __launch_bounds__(kTileRows, 4)
k_propagate_cull(Rows R, const Tile *__restrict__ tiles, const __grid_constant__ CullViews cvw, VisibleBufs vb,
                 DevStats *__restrict__ stats, uint32_t static_opt, uint32_t parity) {
    __shared__ TileSmem s;
    const Tile tile = tiles[blockIdx.x];
    const uint32_t lr = threadIdx.x;
    const bool active = lr < tile.n_rows;
    const uint32_t row = tile.base + lr;

    // ---- phase 1: loads -------------------------------------------------------------
    float4 A = make_float4(0, 0, 0, 0), q = A, bA = A;
    float2 C = make_float2(0, 0), bB = C;
    Aff g;            // current GlobalTransform (old value until overwritten)
    g.r0 = g.r1 = g.r2 = A;
    uint32_t f = 0, st8 = 0, topo = T_DETACHED;
    if (active) {
        f = R.flags[row];
        st8 = R.state[row];
        g.r0 = R.gt0[row]; g.r1 = R.gt1[row]; g.r2 = R.gt2[row];
        if (PROP) { topo = R.topo[row]; A = R.trsA[row]; q = R.trsB[row]; C = R.trsC[row]; }
        if (CULL) { bA = R.bndA[row]; bB = R.bndB[row]; }
    }
    bool visited = false, changed = false;
    if (PROP) {
        const uint32_t depth = (topo >> 9) & 0x1FFu, plocal = topo & 0x1FFu;
        const bool tchanged = f & F_TCHANGED;
        const bool has_children = topo & T_HAS_CHILDREN;
        // -- mark_dirty_trees (systems.rs:111-306) inside the tile: climb the staged parent links
        bool dirty = tchanged;
        if (static_opt && R.dirty != nullptr) {
            dirty = active && R.dirty[row];     // multi-pass plan: k_mark_dirty_global ran first
        } else if (static_opt && tile.n_levels > 1) {
            s.parent[lr] = (uint16_t)((depth > 0) ? plocal : 0xFFFFu);
            s.dirty[lr] = 0;
            __syncthreads();
            if (active && tchanged) {
                uint32_t c = lr;
                while (!s.dirty[c]) {           // benign race: every writer stores 1, every chain finishes
                    s.dirty[c] = 1;
                    const uint32_t p = s.parent[c];
                    if (p == 0xFFFFu) break;
                    c = p;
                }
            }
            __syncthreads();
            dirty = s.dirty[lr];
        }
        const Aff l = affine_from_trs(A, q, C);
        const uint32_t my_level = (active && !(topo & T_DETACHED)) ? depth : 0xFFFFFFFFu;
        // a detached row (ChildOf without a usable parent) is never visited, and neither is its subtree
        if (active && (topo & T_DETACHED) && has_children) s.st[lr] = 0;
        // ---- level 0: roots, flat entities, rows whose parent was finished by an earlier pass
        if (my_level == 0) {
            if (topo & T_ROOT) {
                // flat entity: sync_simple_transforms (systems.rs:42-79); root with children:
                // unconditional write (systems.rs:525-530)
                visited = has_children ? (!static_opt || dirty) : tchanged;
                changed = visited;
                if (changed) g = l;
            } else {
                const uint32_t pr = R.parent[row];
                const uint32_t ps = R.state[pr];
                visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                if (visited) {
                    Aff n;
                    n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                    changed = row_neq(n.r0, g.r0) | row_neq(n.r1, g.r1) | row_neq(n.r2, g.r2);
                    if (changed) g = n;
                }
            }
            if (has_children) {
                s.g0[lr] = g.r0; s.g1[lr] = g.r1; s.g2[lr] = g.r2;
                s.st[lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            }
        }
        // ---- deeper levels: propagate_descendants_unchecked (systems.rs:706-727)
        for (uint32_t lvl = 1; lvl < tile.n_levels; ++lvl) {
            if (lvl < 32u && ((tile.warp_sync_mask >> lvl) & 1u)) __syncwarp(); else __syncthreads();
            if (my_level == lvl) {
                const uint32_t pst = s.st[plocal];
                visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                if (visited) {
                    Aff n;
                    n.r0 = affine_mul_row(s.g0[plocal], l); n.r1 = affine_mul_row(s.g1[plocal], l); n.r2 = affine_mul_row(s.g2[plocal], l);
                    changed = row_neq(n.r0, g.r0) | row_neq(n.r1, g.r1) | row_neq(n.r2, g.r2);   // set_if_neq
                    if (changed) g = n;
                }
                if (has_children) {
                    s.g0[lr] = g.r0; s.g1[lr] = g.r1; s.g2[lr] = g.r2;
                    s.st[lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
                }
            }
        }
        if (active) {
            if (changed) { R.gt0[row] = g.r0; R.gt1[row] = g.r1; R.gt2[row] = g.r2; }
            if (tchanged) R.flags[row] = (uint8_t)(f & ~F_TCHANGED);
        }
    }
    uint32_t out = st8 & (S_VV | S_HAS_CLASS);
    if (PROP) out |= (changed ? S_GT_CHANGED : 0u) | (visited ? S_VISITED : 0u);
    else out |= st8 & (S_GT_CHANGED | S_VISITED);

    // ---- phase 3: cull ----------------------------------------------------------------
    bool vv_changed = false;
    if (CULL) {
        const bool in_query = active && !(f & F_NO_CPU_CULL);          // Without<NoCpuCulling>
        const bool base = in_query && (f & F_INHERITED);
        const bool rej_base = base;
        const uint32_t prev = st8 & 1u;                                // reset_view_visibility: v = (v&1)<<1
        const uint32_t lane = lr & 31u;
        const bool has_aabb = f & F_AABB;
        const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
        // world-space bounding sphere (visibility/mod.rs:825-829): Aabb -> transform_point3a(center),
        // radius_vec3a(half_extents); Sphere -> as stored (or the row's own translation)
        float cx, cy, cz, radius;
        const float hx = bA.w, hy = bB.x, hz = bB.y;
        if (has_aabb) {
            cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
            cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
            cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
            const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
            const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
            const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
            radius = sqrtf((vx * vx + vy * vy) + vz * vz);
        } else {
            const bool from_gt = f & F_SPHERE_GT;
            cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
            radius = bA.w;
        }
        unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
        if (!SIMPLE && active) {
            if (R.layers != nullptr) elayers = R.layers[row];
            if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
            if (R.rank != nullptr) rnk = R.rank[row];
        }
        // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
        const uint32_t rejmask = warp_view_reject(cvw, rej_base && do_test, rej_base && !do_test, cx, cy, cz, radius);
        bool any = false;
        uint32_t my_ballot = 0;
        // The per-view constants arrive as a __grid_constant__ kernel parameter: with the view loop
        // unrolled every plane component is a constant-bank operand of the FMUL/FADD itself (no loads).
#pragma unroll
        for (uint32_t v = 0; v < kMaxViews; ++v) {
            if (v >= cvw.n_views) break;
            const uint32_t von = cvw.on[v];
            if (!(von & 1u)) continue;                                 // !camera.is_active (grid-uniform)
            if (SIMPLE && !(von & 4u)) continue;                       // bit2: the view includes the default layer
            if (((rejmask >> v) & 1u) && !(von & 2u)) continue;         // every row of this warp is outside this view's frustum
            bool vis = base;
            if (!SIMPLE) {
                vis = vis && layers_intersect(R, cvw, row, v, elayers);
                if ((f & F_RANGE) && R.range != nullptr) {
                    const int32_t ri = cvw.range_index[v];
                    vis = vis && ri >= 0 && ((erange >> ri) & 1u);
                }
            }
            if (do_test && !(von & 2u)) {
                // Frustum::intersects_sphere, planes 0..4 (primitives.rs:255-268), branch-free
                const float d0 = plane_dot_point(cvw.planes[v][0], cx, cy, cz), d1 = plane_dot_point(cvw.planes[v][1], cx, cy, cz);
                const float d2 = plane_dot_point(cvw.planes[v][2], cx, cy, cz), d3 = plane_dot_point(cvw.planes[v][3], cx, cy, cz);
                const float d4 = plane_dot_point(cvw.planes[v][4], cx, cy, cz);
                const bool out_s = (d0 + radius <= 0.0f) | (d1 + radius <= 0.0f) | (d2 + radius <= 0.0f) |
                                   (d3 + radius <= 0.0f) | (d4 + radius <= 0.0f);
                vis = vis && !out_s;
                if (vis && has_aabb) {
                    // Frustum::intersects_obb(aabb, affine, true, false) (primitives.rs:272-294);
                    // the plane . (center,1) terms are the ones computed above, bit for bit
                    const float d[5] = {d0, d1, d2, d3, d4};
                    bool out_o = false;
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        const float4 n = cvw.planes[v][k];   // Aabb::relative_radius (primitives.rs:109-119)
                        const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                        const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                        const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                        const float rr = (dx * hx + dy * hy) + dz * hz;
                        out_o |= (d[k] + rr <= 0.0f);
                    }
                    vis = !out_o;
                }
            }
            any |= vis;
            // entities without a VisibilityClass are set_visible() but not listed (mod.rs:846-857)
            const bool listed = vis && (st8 & S_HAS_CLASS);
            if (SIMPLE || R.rank == nullptr) {
                const uint32_t b = __ballot_sync(0xFFFFFFFFu, listed);
                if (lane == v) my_ballot = b;
            } else if (listed) {
                uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
                uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
                atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
            }
        }
        // warp-ballot compaction: lane v publishes view v's 32 bits; 32 consecutive rows touch at
        // most two words of the rank-ordered mask
        if (my_ballot) {
            uint32_t *mask = vb.mask + (size_t)lane * vb.words_stride;
            uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride;
            const uint32_t row0 = row - lane, w0 = row0 >> 5, sh = row0 & 31u;
            const uint32_t lo = my_ballot << sh, hi = sh ? (my_ballot >> (32u - sh)) : 0u;
            if (lo) { atomicOr(mask + w0, lo); atomicAdd(cc + (w0 / kChunkWords), __popc(lo)); }
            if (hi) { atomicOr(mask + w0 + 1, hi); atomicAdd(cc + ((w0 + 1) / kChunkWords), __popc(hi)); }
        }
        if (in_query) {
            // set_visible + mark_newly_hidden_entities_invisible (mod.rs:292-306, 908-918):
            // visible -> 0b01 | prev<<1 ; hidden -> 0 ; Changed fires on 0->1 and 1->0 only
            out = (out & ~S_VV) | (any ? (1u | (prev << 1)) : 0u);
            vv_changed = (any ? 1u : 0u) != prev;
            if (vv_changed) out |= S_VV_CHANGED;
        }
    } else {
        out |= st8 & S_VV_CHANGED;
    }
    if (active && out != st8) R.state[row] = (uint8_t)out;

    // per-frame change counters (one atomic per CTA)
    const int n_gt = __syncthreads_count(PROP && changed);
    const int n_vv = __syncthreads_count(vv_changed);
    if (lr == 0) {
        if (n_gt) atomicAdd(&stats->changed[parity][0], (uint32_t)n_gt);
        if (n_vv) atomicAdd(&stats->changed[parity][1], (uint32_t)n_vv);
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 1b: the same fused propagate -> cull tile pass as a PERSISTENT, TMA-staged kernel.
//
// One CTA per SM slot loops over tiles.  A tile's columns (Transform, old GlobalTransform, bounds,
// topo, flags, state: 11 arrays, 118 B/row) are pulled into shared memory with cp.async.bulk (the
// TMA engine, SASS UBLKCP) by ONE elected thread and land on an mbarrier; two stages are kept, so
// the next tile's 30 KB are in flight while the current tile is computed.  That takes the global
// loads and their address arithmetic out of the 256 compute threads, keeps >= 2 tiles of loads
// per CTA in flight independent of occupancy, and lets the hierarchy walk update the
// GlobalTransform tile IN PLACE in shared memory: a child reads its parent's row of the tile
// (already new if it changed, still the old bits if set_if_neq kept it), and the finished tile
// goes back to HBM with one bulk store per matrix row array.
// Bulk copies need 16-byte aligned addresses and sizes: the window is [base & ~15, round_up16(base + n)),
// so every array's byte range is 16 B aligned whatever the element size; arrays carry 32 rows of padding.
// ------------------------------------------------------------------------------------------
constexpr int kWin = kTileRows + 16;     // rows per staged window (base misalignment <= 15)

struct __align__(128) TileStage {
    float4 trsA[kWin], trsB[kWin];
    float4 gt0[kWin], gt1[kWin], gt2[kWin];
    float2 trsC[kWin];
    uint32_t topo[kWin];
    uint8_t flags[kWin], state[kWin];
};
struct TmaSmem {
    TileStage st[2];
    unsigned long long bar[2];       // full[s]: the tile's columns have landed in stage s (TMA complete_tx)
    unsigned long long walked[2];    // walked[s]: all 8 warps are done walking the tile in stage s, hold their rows in registers,
                                     //            and have looked at the NEXT tile's change flags (climb[s ^ 1] is final)
    uint32_t next_tile[2];           // k_propagate_cull_tma: the tile this CTA processes after the one in stage s
    uint32_t climb[2];               // climb[s] == it: a non-root row of the tile of iteration it (stage s) has Changed<Transform>
    uint16_t parent[kTileRows];
    uint8_t pst[kTileRows];      // bit0 visited, bit1 gt changed
    uint8_t dirty[kTileRows];
};

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// the same wait with a watchdog: a hand-over that never comes (a protocol bug) traps -- the launch fails -- instead of hanging the GPU
__device__ __forceinline__ void mbar_wait_guarded(unsigned long long *bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) break;
        if (++spins > (1u << 24)) __trap();
    }
}
__device__ __forceinline__ void mbar_arrive_cta(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}

template <bool PROP, bool CULL>
__device__ __forceinline__ void issue_tile_loads(const Rows &R, const Tile &t, TileStage &S, unsigned long long *bar) {
    const uint32_t a = t.base & ~15u;
    const uint32_t cnt = ((t.base - a) + t.n_rows + 15u) & ~15u;
    uint32_t bytes = cnt * (48u + 2u);
    if (PROP) bytes += cnt * (40u + 4u);
    mbar_expect_tx(bar, bytes);
    bulk_g2s(S.gt0, R.gt0 + a, cnt * 16u, bar); bulk_g2s(S.gt1, R.gt1 + a, cnt * 16u, bar); bulk_g2s(S.gt2, R.gt2 + a, cnt * 16u, bar);
    bulk_g2s(S.flags, R.flags + a, cnt, bar); bulk_g2s(S.state, R.state + a, cnt, bar);
    if (PROP) {
        bulk_g2s(S.trsA, R.trsA + a, cnt * 16u, bar); bulk_g2s(S.trsB, R.trsB + a, cnt * 16u, bar);
        bulk_g2s(S.trsC, R.trsC + a, cnt * 8u, bar); bulk_g2s(S.topo, R.topo + a, cnt * 4u, bar);
    }
}

#ifdef B200VIS_TILE_TIMING
// debug build only (tools/tile_timing.py): per-CTA phase timestamps of the tile kernel, read back through
// b200vis_debug_tile_timing; not compiled into the product library
__device__ unsigned long long g_tile_timing[8192 * 16];
#define TT(slot) do { if (lr == 0 && blockIdx.x < 8192u) g_tile_timing[blockIdx.x * 16u + (slot)] = clock64(); } while (0)
#define TTW(slot) do { if (lr == 224u && blockIdx.x < 8192u) g_tile_timing[blockIdx.x * 16u + (slot)] = clock64(); } while (0)
#else
#define TT(slot) do { } while (0)
#define TTW(slot) do { } while (0)
#endif
template <bool PROP, bool CULL, bool SIMPLE>
__global__ void __launch_bounds__(kTileRows, 4)
k_propagate_cull_tma(Rows R, const Tile *__restrict__ tiles, uint32_t n_tiles, const __grid_constant__ CullViews cvw,
                     VisibleBufs vb, DevStats *__restrict__ stats, uint32_t static_opt, uint32_t parity,
                     uint32_t *__restrict__ ticket, uint32_t ticket_base) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    TmaSmem &s = *reinterpret_cast<TmaSmem *>(smem_raw);
    const uint32_t lr = threadIdx.x;
    if (lr == 0) {
        mbar_init(&s.bar[0], 1); mbar_init(&s.bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // launched with programmatic stream serialization: everything above overlapped the previous kernel's tail
    TT(0);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    TT(1);
    uint32_t t = blockIdx.x;
    if (lr == 0 && t < n_tiles) issue_tile_loads<PROP, CULL>(R, tiles[t], s.st[0], &s.bar[0]);
    uint32_t n_gt_total = 0, n_vv_total = 0;
    // Tile hand-out: a CTA starts on tile blockIdx.x and then takes the tiles the grid has not started yet in ticket order
    // (one atomic per tile, drawn by thread 0 when it prefetches, i.e. one tile ahead).  A fixed stride would leave a CTA with
    // ceil(n/g) tiles running next to finished neighbours with floor(n/g) -- a fifth of the pass at 3.3 tiles per CTA.  The
    // ticket counter is never reset: every launch draws exactly n_tiles tickets, and the host passes the running base.
    for (uint32_t it = 0; t < n_tiles; ++it) {
        const uint32_t sidx = it & 1u;
        const Tile tile = tiles[t];
        mbar_wait(&s.bar[sidx], (it >> 1) & 1u);
        if (it == 1) { TT(2); }
        TileStage &S = s.st[sidx];
        const uint32_t off = tile.base & 15u;
        const uint32_t li = off + lr;                 // index into the staged window
        const bool active = lr < tile.n_rows;
        const uint32_t row = tile.base + lr;
        const uint32_t f = active ? S.flags[li] : 0u;
        const uint32_t st8 = active ? S.state[li] : 0u;
        // bounds are only needed after the hierarchy walk: plain coalesced loads issued now, consumed in phase 3
        // (keeping them out of the staged window lets a fourth CTA fit in shared memory)
        float4 bA = make_float4(0, 0, 0, 0); float2 bB = make_float2(0, 0);
        if (CULL && active) { bA = R.bndA[row]; bB = R.bndB[row]; }

        bool visited = false, changed = false;
        if (PROP) {
            const uint32_t topo = active ? S.topo[li] : T_DETACHED;
            const uint32_t depth = (topo >> 9) & 0x1FFu, plocal = topo & 0x1FFu;
            const bool tchanged = f & F_TCHANGED;
            const bool has_children = topo & T_HAS_CHILDREN;
            bool dirty = tchanged;
            if (static_opt && R.dirty != nullptr) {
                dirty = active && R.dirty[row];
            } else if (static_opt && tile.n_levels > 1 && __syncthreads_or(tchanged && depth > 0)) {
                // only when a non-root row of the tile changed does anything have to climb: otherwise every row's
                // TransformTreeChanged bit equals its own Changed<Transform> bit (one barrier instead of two + a climb)
                s.parent[lr] = (uint16_t)((depth > 0) ? plocal : 0xFFFFu);
                s.dirty[lr] = 0;
                __syncthreads();
                if (active && tchanged) {
                    uint32_t c = lr;
                    while (!s.dirty[c]) {
                        s.dirty[c] = 1;
                        const uint32_t p = s.parent[c];
                        if (p == 0xFFFFu) break;
                        c = p;
                    }
                }
                __syncthreads();
                dirty = s.dirty[lr];
            }
            if (it == 1) { TT(3); }    // dirty phase done
            const Aff l = affine_from_trs(S.trsA[li], S.trsB[li], S.trsC[li]);
            const uint32_t my_level = (active && !(topo & T_DETACHED)) ? depth : 0xFFFFFFFFu;
            if (active && (topo & T_DETACHED) && has_children) s.pst[lr] = 0;
            if (my_level == 0) {
                Aff n = l;
                if (topo & T_ROOT) {
                    visited = has_children ? (!static_opt || dirty) : tchanged;
                    changed = visited;
                } else {
                    const uint32_t pr = R.parent[row];
                    const uint32_t ps = R.state[pr];
                    visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                    if (visited) {
                        n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                        changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);
                    }
                }
                if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                if (has_children) s.pst[lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            }
            if (it == 1) { TT(4); }    // local affine + level 0 done
            // one level of the walk for this thread's row: the parent's rows are the tile's own (in-place) GlobalTransform entries
            auto walk_row = [&]() {
                const uint32_t pst = s.pst[plocal];
                const uint32_t pi = off + plocal;
                visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                if (visited) {
                    Aff n;
                    n.r0 = affine_mul_row(S.gt0[pi], l); n.r1 = affine_mul_row(S.gt1[pi], l); n.r2 = affine_mul_row(S.gt2[pi], l);
                    changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);   // set_if_neq
                    if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                }
                if (has_children) s.pst[lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            };
            if (tile.lvl_warps != 0ull) {
                // Per-warp level schedule (2..8 levels).  A warp only takes part in the hand-over of the levels its own rows
                // produce (level l-1) or consume (level l), through hardware named barrier l with exactly the warps the planner
                // counted (Tile::lvl_warps): consumers bar.sync, pure producers bar.arrive and go on; a leaf warp waits once
                // instead of once per level, and nobody pays the loop for levels that are not theirs.  (The tile still ends in a
                // CTA-wide barrier, so one set of barrier ids is enough here.)
                // (a detached row takes no part in the walk but publishes pst = 0 for its children: it counts as a level-0 row)
                const uint32_t lmask = __reduce_or_sync(0xFFFFFFFFu, active ? (1u << (depth & 15u)) : 0u);
                uint32_t need = (lmask | (lmask << 1)) & ((1u << tile.n_levels) - 2u);
                while (need) {
                    const uint32_t lvl = (uint32_t)__ffs((int)need) - 1u;
                    need &= need - 1u;
                    const bool consumer = (lmask >> lvl) & 1u;
                    if ((tile.warp_sync_mask >> lvl) & 1u) {       // every edge into this level stays inside a warp
                        if (!consumer) continue;
                        __syncwarp();
                    } else {
                        const uint32_t cnt = ((uint32_t)(tile.lvl_warps >> (4u * lvl)) & 15u) * 32u;
                        if (!consumer) {
                            __threadfence_block();
                            asm volatile("bar.arrive %0, %1;" ::"r"(lvl), "r"(cnt) : "memory");
                            continue;
                        }
                        asm volatile("bar.sync %0, %1;" ::"r"(lvl), "r"(cnt) : "memory");
                    }
                    if (my_level == lvl) walk_row();
                }
            } else {
                for (uint32_t lvl = 1; lvl < tile.n_levels; ++lvl) {
                    if (lvl < 32u && ((tile.warp_sync_mask >> lvl) & 1u)) __syncwarp(); else __syncthreads();
                    if (my_level == lvl) walk_row();
                    if (it == 1 && lvl <= 7) { TT(4 + lvl); }   // thread 0 after the level's barrier and (for level-lvl rows) work
                }
            }
            if (active && tchanged) R.flags[row] = (uint8_t)(f & ~F_TCHANGED);
        }
        if (it == 1) { TT(12); }   // walk done
        // Prefetch the NEXT tile into the other stage.  That stage was last read by the previous tile's bulk store,
        // issued most of an iteration ago, so the wait below is (almost always) already satisfied: putting the
        // prefetch here instead of at the top of the loop keeps the store drain off every warp's critical path.
        if (lr == 0) {
            const uint32_t tn = ticket ? gridDim.x + (atomicAdd(ticket, 1u) - ticket_base) : t + gridDim.x;
            if (tn < n_tiles) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                issue_tile_loads<PROP, CULL>(R, tiles[tn], s.st[sidx ^ 1u], &s.bar[sidx ^ 1u]);
            }
            s.next_tile[sidx] = tn;      // read by everybody behind the tile's closing barrier
        }
        uint32_t out = st8 & (S_VV | S_HAS_CLASS);
        if (PROP) out |= (changed ? S_GT_CHANGED : 0u) | (visited ? S_VISITED : 0u);
        else out |= st8 & (S_GT_CHANGED | S_VISITED);

        bool vv_changed = false;
        if (CULL) {
            Aff g; g.r0 = S.gt0[li]; g.r1 = S.gt1[li]; g.r2 = S.gt2[li];   // own row: written by this thread or untouched
            const bool in_query = active && !(f & F_NO_CPU_CULL);
            const bool base = in_query && (f & F_INHERITED);
        const bool rej_base = base;
            const uint32_t prev = st8 & 1u;
            const uint32_t lane = lr & 31u;
            const bool has_aabb = f & F_AABB;
            const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
            float cx, cy, cz, radius;
            const float hx = bA.w, hy = bB.x, hz = bB.y;
            if (has_aabb) {
                cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
                cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
                cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
                const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
                const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
                const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
                radius = sqrtf((vx * vx + vy * vy) + vz * vz);
            } else {
                const bool from_gt = f & F_SPHERE_GT;
                cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
                radius = bA.w;
            }
            unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
            if (!SIMPLE && active) {
                if (R.layers != nullptr) elayers = R.layers[row];
                if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
                if (R.rank != nullptr) rnk = R.rank[row];
            }
            // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
            const uint32_t rejmask = warp_view_reject(cvw, rej_base && do_test, rej_base && !do_test, cx, cy, cz, radius);
            bool any = false;
            uint32_t my_ballot = 0;
#pragma unroll
            for (uint32_t v = 0; v < kMaxViews; ++v) {
                if (v >= cvw.n_views) break;
                const uint32_t von = cvw.on[v];
                if (!(von & 1u)) continue;
                if (SIMPLE && !(von & 4u)) continue;   // bit2: the view includes the default layer
                if (((rejmask >> v) & 1u) && !(von & 2u)) continue;         // every row of this warp is outside this view's frustum
                bool vis = base;
                if (!SIMPLE) {
                    vis = vis && layers_intersect(R, cvw, row, v, elayers);
                    if ((f & F_RANGE) && R.range != nullptr) {
                        const int32_t ri = cvw.range_index[v];
                        vis = vis && ri >= 0 && ((erange >> ri) & 1u);
                    }
                }
                if (do_test && !(von & 2u)) {
                    const float d0 = plane_dot_point(cvw.planes[v][0], cx, cy, cz), d1 = plane_dot_point(cvw.planes[v][1], cx, cy, cz);
                    const float d2 = plane_dot_point(cvw.planes[v][2], cx, cy, cz), d3 = plane_dot_point(cvw.planes[v][3], cx, cy, cz);
                    const float d4 = plane_dot_point(cvw.planes[v][4], cx, cy, cz);
                    const bool out_s = (d0 + radius <= 0.0f) | (d1 + radius <= 0.0f) | (d2 + radius <= 0.0f) |
                                       (d3 + radius <= 0.0f) | (d4 + radius <= 0.0f);
                    vis = vis && !out_s;
                    if (vis && has_aabb) {
                        const float d[5] = {d0, d1, d2, d3, d4};
                        bool out_o = false;
#pragma unroll
                        for (int k = 0; k < 5; ++k) {
                            const float4 n = cvw.planes[v][k];
                            const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                            const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                            const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                            const float rr = (dx * hx + dy * hy) + dz * hz;
                            out_o |= (d[k] + rr <= 0.0f);
                        }
                        vis = !out_o;
                    }
                }
                any |= vis;
                const bool listed = vis && (st8 & S_HAS_CLASS);
                if (SIMPLE || R.rank == nullptr) {
                    const uint32_t b = __ballot_sync(0xFFFFFFFFu, listed);
                    if (lane == v) my_ballot = b;
                } else if (listed) {
                    uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
                    uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
                    atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                    atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
                }
            }
            if (my_ballot) {
                uint32_t *mask = vb.mask + (size_t)lane * vb.words_stride;
                uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride;
                const uint32_t row0 = row - lane, w0 = row0 >> 5, sh = row0 & 31u;
                const uint32_t lo = my_ballot << sh, hi = sh ? (my_ballot >> (32u - sh)) : 0u;
                if (lo) { atomicOr(mask + w0, lo); atomicAdd(cc + (w0 / kChunkWords), __popc(lo)); }
                if (hi) { atomicOr(mask + w0 + 1, hi); atomicAdd(cc + ((w0 + 1) / kChunkWords), __popc(hi)); }
            }
            if (in_query) {
                out = (out & ~S_VV) | (any ? (1u | (prev << 1)) : 0u);
                vv_changed = (any ? 1u : 0u) != prev;
                if (vv_changed) out |= S_VV_CHANGED;
            }
        } else {
            out |= st8 & S_VV_CHANGED;
        }
        if (active && out != st8) R.state[row] = (uint8_t)out;
        // a light row publishes what assign_objects_to_clusters needs of it (GlobalTransform::translation,
        // ViewVisibility::get) so that the cluster kernels never touch the row arrays again
        if (CULL && R.light_snap != nullptr && (f & F_SPHERE_GT) && active) {
            const uint32_t ord = R.light_ord[row];     // 0xFFFFFFFF: a sphere-from-GT row that is not a current light
            if (ord < R.n_lights) R.light_snap[ord] = make_float4(S.gt0[li].w, S.gt1[li].w, S.gt2[li].w, (out & 1u) ? 1.0f : 0.0f);
        }

        // end of tile: everybody is done with this stage; count changes; write the tile's matrices back
        n_gt_total += (PROP && changed) ? 1u : 0u;      // per-thread tallies, reduced once at the end of the kernel
        n_vv_total += vv_changed ? 1u : 0u;
        if (it == 1) { TT(13); }   // cull done
        const int any_gt = __syncthreads_or(PROP && changed);
        if (it == 1) { TT(15); }
        t = s.next_tile[sidx];
        if (lr == 0) {
            if (PROP && any_gt) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic smem writes -> async proxy
                const uint32_t bytes = (uint32_t)tile.n_rows * 16u;
                bulk_s2g(R.gt0 + tile.base, S.gt0 + off, bytes); bulk_s2g(R.gt1 + tile.base, S.gt1 + off, bytes);
                bulk_s2g(R.gt2 + tile.base, S.gt2 + off, bytes);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    if (lr == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    TT(14);
    // block-reduce the per-thread tallies (warp shuffle, then one shared-memory atomic per warp)
    __shared__ uint32_t s_cnt[2];
    if (lr < 2) s_cnt[lr] = 0;
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { n_gt_total += __shfl_xor_sync(0xFFFFFFFFu, n_gt_total, o); n_vv_total += __shfl_xor_sync(0xFFFFFFFFu, n_vv_total, o); }
    if ((lr & 31u) == 0) { if (n_gt_total) atomicAdd(&s_cnt[0], n_gt_total); if (n_vv_total) atomicAdd(&s_cnt[1], n_vv_total); }
    __syncthreads();
    if (lr == 0) {
        if (s_cnt[0]) atomicAdd(&stats->changed[parity][0], s_cnt[0]);
        if (s_cnt[1]) atomicAdd(&stats->changed[parity][1], s_cnt[1]);
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 1L (the DEFAULT tile kernel; B200VIS_TILE_KERNEL=tma selects 1b): kernel 1b on an instruction and exposed-latency diet.
// ncu's source view of 1b (profiles/r02b_tma_basic_blocks.txt) shows ~820 warp instructions per 32 rows of which half are
// bookkeeping, an SM that issues ~2 warp instructions per cycle whatever the occupancy (DESIGN.md section 7), and four places where
// a long latency is exposed on every tile:
//   * the tile descriptor (LDG of tiles[t]) at the top of a tile                  -> descriptors travel through shared memory:
//     the bookkeeping thread fetches the descriptor of the CTA's tile i+2 with cp.async while tile i is culled;
//   * the TMA prefetch of tile i+1 is issued after the walk of tile i by thread 0 (the warp every level of the walk waits
//     for), behind a dependent ticket atomic + descriptor load                    -> the bookkeeping thread is the LAST thread
//     (a leaf warp that idles while the levels above it are walked), the ticket is drawn one tile further ahead and the
//     prefetch goes out at the top of the tile, a whole walk earlier;
//   * the view-rejection test reads its planes with register-indexed LDC          -> planes are staged in shared memory once
//     per CTA; the box is built with f32 warp reductions (CREDUX.F32) instead of order-preserving integer transforms;
//   * the per-view loop was unrolled 8x with the plane operands in the constant bank (48 KB of code, a test + branch per
//     view even when the warp rejected it)                                         -> one rolled loop over the set bits of
//     (active views & ~rejected), planes from shared memory: a warp that rejects every view skips the loop in 3 instructions.
// On top of that: the tile's top levels are walked in registers with warp shuffles; B200VIS_LEAN_PROBE=8 bounds the warp's rows
// with a sphere (3 shuffles + 1 reduction) instead of a box (7 reductions) in the warp-level view rejection (measured: +1 %).
// Same results bit for bit (tests/test_gpu_bench_scale.py runs the bench workload through it).
// ------------------------------------------------------------------------------------------
// MINB = 4: the whole tile (Transform, GlobalTransform, topo, flags, state: 94 B/row) is staged in both stages, as in kernel 1b.
// MINB = 5, 6: Transform stays out of the staged window (54 B/row staged) -- it is consumed in the first hundred instructions of a
// tile, so it comes in through plain coalesced loads issued above the wait for the tile (the bookkeeping thread has pulled the
// columns into L2 a tile ahead) -- which lets a 5th / 6th CTA fit an SM's shared memory; the register budget (48 / 40) is met with
// a handful of spills, and the named level barriers use immediate ids so that a CTA owns 8 of the SM's hardware barriers, not 16.
template <bool WITH_TRS> struct __align__(128) LeanStage;
template <> struct __align__(128) LeanStage<true> {
    float4 gt0[kWin], gt1[kWin], gt2[kWin];
    uint32_t topo[kWin];
    uint8_t flags[kWin], state[kWin];
    float4 trsA[kWin], trsB[kWin];
    float2 trsC[kWin];
};
template <> struct __align__(128) LeanStage<false> {
    float4 gt0[kWin], gt1[kWin], gt2[kWin];
    uint32_t topo[kWin];
    uint8_t flags[kWin], state[kWin];
};
template <bool WITH_TRS>
struct LeanSmem {
    LeanStage<WITH_TRS> st[2];
    unsigned long long bar[2];       // full[s]: the tile's columns have landed in stage s
    Tile tdesc[3];                   // descriptor of the CTA's i-th tile in slot i % 3 (i+2 is fetched while i is processed)
    uint32_t next_tile[2];
    float4 vplanes[kMaxViews * 5];   // the views' culling planes, [view][L,R,T,B,Near]
    float vlen[kMaxViews * 5];       // |normal| of each plane, rounded up (1 for normalised half spaces)
    unsigned long long done[2];      // PIPE: all 8 warps are through with the tile in stage s (one arrival per warp)
    uint32_t anyflag[2];             // PIPE: some row of the tile in stage s got a new GlobalTransform (the stage has to be stored)
    uint16_t parent[kTileRows];
    uint8_t pst[2][kTileRows];       // bit0 visited, bit1 gt changed; PIPE: one copy per stage, else copy 0
    uint8_t dirty[kTileRows];
};
template <bool PROP, bool CULL, bool WITH_TRS>
__device__ __forceinline__ void issue_lean_loads(const Rows &R, const Tile &t, LeanStage<WITH_TRS> &S, unsigned long long *bar) {
    const uint32_t a = t.base & ~15u;
    const uint32_t cnt = ((t.base - a) + t.n_rows + 15u) & ~15u;
    uint32_t bytes = cnt * (48u + 2u);
    if (PROP) bytes += cnt * 4u;
    if (PROP && WITH_TRS) bytes += cnt * 40u;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(S.gt0, R.gt0 + a, cnt * 16u, bar); bulk_g2s(S.gt1, R.gt1 + a, cnt * 16u, bar); bulk_g2s(S.gt2, R.gt2 + a, cnt * 16u, bar);
    bulk_g2s(S.flags, R.flags + a, cnt, bar); bulk_g2s(S.state, R.state + a, cnt, bar);
    if (PROP) bulk_g2s(S.topo, R.topo + a, cnt * 4u, bar);
    if constexpr (WITH_TRS) {
        if (PROP) {
            bulk_g2s(S.trsA, R.trsA + a, cnt * 16u, bar); bulk_g2s(S.trsB, R.trsB + a, cnt * 16u, bar);
            bulk_g2s(S.trsC, R.trsC + a, cnt * 8u, bar);
        }
    } else if (PROP) {     // the Transform columns of that tile into L2: its rows load them straight into registers
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(R.trsA + a), "r"(cnt * 16u) : "memory");
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(R.trsB + a), "r"(cnt * 16u) : "memory");
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(R.trsC + a), "r"(cnt * 8u) : "memory");
    }
}
// hardware named barrier `id` (1..7) with IMMEDIATE ids: ptxas then counts 8 barriers per CTA instead of assuming all 16 (the SM
// has 64, i.e. 16 per CTA cap residency at 4 CTAs).  Seven predicated barrier instructions, no jump table: this sits on the walk's
// critical path and every instruction here has a fixed latency.
#define B200VIS_BAR_SEQ(OP) \
    "{\n.reg .pred p;\n" \
    "setp.eq.u32 p, %0, 1;\n@p " OP " 1, %1;\n" "setp.eq.u32 p, %0, 2;\n@p " OP " 2, %1;\n" "setp.eq.u32 p, %0, 3;\n@p " OP " 3, %1;\n" \
    "setp.eq.u32 p, %0, 4;\n@p " OP " 4, %1;\n" "setp.eq.u32 p, %0, 5;\n@p " OP " 5, %1;\n" "setp.eq.u32 p, %0, 6;\n@p " OP " 6, %1;\n" \
    "setp.ge.u32 p, %0, 7;\n@p " OP " 7, %1;\n}\n"
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t cnt) { asm volatile(B200VIS_BAR_SEQ("bar.sync") ::"r"(id), "r"(cnt) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t cnt) { asm volatile(B200VIS_BAR_SEQ("bar.arrive") ::"r"(id), "r"(cnt) : "memory"); }
#undef B200VIS_BAR_SEQ
__device__ __forceinline__ float redux_min_f32(float x) { float r; asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float redux_max_f32(float x) { float r; asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ void cp_async_tile_desc(Tile *dst, const Tile *src) {     // 24 bytes, 8-byte aligned on both sides
    const uint32_t d = smem_u32(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(src) : "memory");
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d + 8u), "l"(reinterpret_cast<const uint8_t *>(src) + 8) : "memory");
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d + 16u), "l"(reinterpret_cast<const uint8_t *>(src) + 16) : "memory");
}
// warp_view_reject with the planes in shared memory and f32 warp reductions; lane = plane * 6 + view, so that the ballot folds
// into one bit per view with four shifts.  Returns a bit per view (views 6 and 7 are never rejected here).
__device__ __forceinline__ uint32_t warp_view_reject_lean(const float4 *vplanes, uint32_t n_views, bool testable, bool blocks,
                                                          float cx, float cy, float cz, float radius) {
    const float inf = __int_as_float(0x7f800000);
    const bool fin = testable && isfinite(((cx + cy) + cz) + radius);
    if (__any_sync(0xFFFFFFFFu, blocks || (testable && !fin))) return 0u;
    const float x0 = redux_min_f32(fin ? cx : inf), x1 = redux_max_f32(fin ? cx : -inf);
    const float y0 = redux_min_f32(fin ? cy : inf), y1 = redux_max_f32(fin ? cy : -inf);
    const float z0 = redux_min_f32(fin ? cz : inf), z1 = redux_max_f32(fin ? cz : -inf);
    const float r1 = redux_max_f32(fin ? radius : -inf);
    if (!(x0 <= x1)) return 0xFFu;                // no frustum-tested row in this warp (and none that blocks): nothing can be visible
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t k = (lane * 43u) >> 8, v = lane - 6u * k;      // k = lane / 6 (lane < 32), v = lane % 6
    bool rej = false;
    if (v < n_views && lane < 30u) {
        const float4 n = vplanes[v * 5u + k];
        const float m = ((fmaxf(n.x * x0, n.x * x1) + fmaxf(n.y * y0, n.y * y1)) + fmaxf(n.z * z0, n.z * z1)) + n.w;
        const float mag = ((fabsf(n.x) * fmaxf(fabsf(x0), fabsf(x1)) + fabsf(n.y) * fmaxf(fabsf(y0), fabsf(y1))) +
                           fabsf(n.z) * fmaxf(fabsf(z0), fabsf(z1))) + (fabsf(n.w) + fabsf(r1));
        rej = (m + r1) + (1e-5f * mag + 1e-6f) < 0.0f;     // ~25x the rounding any exact plane_dot_point(..) + radius can carry
    }
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, rej);
    return (b | (b >> 6) | (b >> 12) | (b >> 18) | (b >> 24)) & 0x3Fu;
}

// The same shortcut with a bounding SPHERE instead of a box: centre c0 = the bounding-sphere centre of the warp's first frustum-tested
// row, radius Rmax = max over its rows of |c_i - c0|_1 + r_i (the 1-norm bounds the 2-norm from above and needs no square root).
// For a plane (n, w): n.c_i + w + r_i <= n.c0 + w + |n| * Rmax, so a plane the sphere is behind -- by the same float margin as
// above, `len` being max(|n| rounded up, 1) (1 for Bevy's normalised half spaces) -- has every row of the warp behind it in
// Frustum::intersects_sphere.  Looser than the box by at most sqrt(3) in radius, a third of the instructions: 3 shuffles and one
// warp reduction instead of seven reductions.  vlen[v * 5 + k] = |n| of plane k of view v (staged once per CTA).
__device__ __forceinline__ uint32_t warp_view_reject_sphere(const float4 *vplanes, const float *vlen, uint32_t n_views, bool testable, bool blocks,
                                                            float cx, float cy, float cz, float radius) {
    const bool fin = testable && isfinite(((cx + cy) + cz) + radius);
    if (__any_sync(0xFFFFFFFFu, blocks || (testable && !fin))) return 0u;
    const uint32_t have = __ballot_sync(0xFFFFFFFFu, fin);
    if (!have) return 0xFFu;                      // no frustum-tested row in this warp (and none that blocks): nothing can be visible
    const int src = __ffs((int)have) - 1;
    const float x0 = __shfl_sync(0xFFFFFFFFu, cx, src), y0 = __shfl_sync(0xFFFFFFFFu, cy, src), z0 = __shfl_sync(0xFFFFFFFFu, cz, src);
    const float mine = ((fabsf(cx - x0) + fabsf(cy - y0)) + fabsf(cz - z0)) + fabsf(radius);
    const float rmax = redux_max_f32(fin ? mine : 0.0f);
    if (!isfinite(rmax)) return 0u;               // (differences of huge finite centres)
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t k = (lane * 43u) >> 8, v = lane - 6u * k;      // k = lane / 6 (lane < 32), v = lane % 6
    bool rej = false;
    if (v < n_views && lane < 30u) {
        const float4 n = vplanes[v * 5u + k];
        const float reach = vlen[v * 5u + k] * rmax;
        const float d = ((n.x * x0 + n.y * y0) + n.z * z0) + n.w;
        const float mag = ((fabsf(n.x * x0) + fabsf(n.y * y0)) + fabsf(n.z * z0)) + (fabsf(n.w) + reach);
        rej = (d + reach) + (1e-5f * mag + 1e-6f) < 0.0f;      // ~25x the rounding of either side
    }
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, rej);
    return (b | (b >> 6) | (b >> 12) | (b >> 18) | (b >> 24)) & 0x3Fu;
}

// PIPE (PROP && CULL, MINB == 4; host side: every tile of the launch is flat or walks with named level barriers): the CTA's warps
// are NOT held together at tile boundaries.  What bounds a tile's time is the longest dependent instruction stream through it
// (a warp issues an instruction every ~7 cycles here whatever the occupancy: ncu r02, probes in DESIGN.md section 7): prologue ->
// top levels (warp 0) -> level K .. 7 hand-overs -> the leaf warps' cull -> closing barrier.  Without the closing barrier, warp 0
// starts the next tile's top levels while the leaf warps still cull this one, and the chain of tile k+1 runs under the cull of tile
// k.  Protocol: a warp that is through with a tile arrives on done[stage] (mbarrier, 8 arrivals) and moves on; only the bookkeeping
// thread waits for it, stores the stage and reloads it with the tile after next.  A tile is loaded after every warp has left the
// tile two before it, so the warps of a CTA are never more than one tile apart: everything per-tile exists twice (stages, pst, the
// named barrier ids lvl + 8 * stage, done, anyflag).  The next tile index travels with the TMA barrier (written before the
// arrive.expect_tx that releases it; "no more tiles" is an arrive without bytes).  mark_dirty_trees' "did a non-root row change"
// is answered by every warp for itself from the staged flags (8 rows per lane) instead of a CTA-wide vote.
template <bool PROP, bool CULL, bool SIMPLE, int MINB, bool PIPE = false>
__global__ void __launch_bounds__(kTileRows, MINB)
k_propagate_cull_lean(Rows R, const Tile *__restrict__ tiles, uint32_t n_tiles, const __grid_constant__ CullViews cvw,
                      VisibleBufs vb, DevStats *__restrict__ stats, uint32_t static_opt, uint32_t parity,
                      uint32_t *__restrict__ ticket, uint32_t ticket_base, uint32_t warp_flip) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    constexpr bool WITH_TRS = MINB <= 4;
    LeanSmem<WITH_TRS> &s = *reinterpret_cast<LeanSmem<WITH_TRS> *>(smem_raw);
    // warp_flip = 0xE0 reverses the order of the CTA's warps (thread t works as logical thread t ^ 0xE0): the rows of a tile's top
    // levels -- the serial chain every other warp waits for -- then sit in the CTA's LAST hardware warp, which the SM's issue
    // arbiter prefers (highest warp id first) when several warps are eligible
    const uint32_t lr = threadIdx.x ^ (warp_flip & 0xE0u);
    const uint32_t probe = warp_flip >> 8;     // bits 0-1: timing probes (results are WRONG): 1 = no level hand-overs at all, 2 = none for levels 1..4; bit 2: top levels through the level loop, bit 3: sphere instead of box in the warp-level view rejection (A/B switches, correct results)
    const bool keeper = lr == (uint32_t)kTileRows - 1u;      // the bookkeeping thread: tickets, descriptors, TMA loads and stores
    static_assert(!PIPE || (PROP && CULL && MINB == 4), "PIPE needs the fused pass with staged Transforms");
    if (keeper) {
        mbar_init(&s.bar[0], 1); mbar_init(&s.bar[1], 1);
        mbar_init(&s.done[0], kTileRows / 32); mbar_init(&s.done[1], kTileRows / 32);
        s.anyflag[0] = 0; s.anyflag[1] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // per-launch view constants: planes into shared memory, the "which views does a row have to be tested against" masks
    uint32_t v_on = 0, v_nofr = 0;
    if (CULL) {
        if (lr < (uint32_t)kMaxViews * 5u) {
            const float4 pl = cvw.planes[lr / 5u][lr % 5u];
            s.vplanes[lr] = pl;
            s.vlen[lr] = fmaxf(sqrtf((pl.x * pl.x + pl.y * pl.y) + pl.z * pl.z) * 1.000001f, 1.0f);   // >= 1: it also scales the rows' own radii
        }
#pragma unroll
        for (uint32_t v = 0; v < (uint32_t)kMaxViews; ++v) {
            if (v < cvw.n_views) {
                const uint32_t on = cvw.on[v];
                if ((on & 1u) && (!SIMPLE || (on & 4u))) v_on |= 1u << v;       // active camera (SIMPLE: whose layers hold the default layer)
                if (on & 2u) v_nofr |= 1u << v;                                  // NoCpuCulling camera: no frustum test
            }
        }
    }
    // launched with programmatic stream serialization: everything above overlapped the previous kernel's tail
    asm volatile("griddepcontrol.wait;" ::: "memory");
    uint32_t t = blockIdx.x;
    uint32_t k_next = n_tiles;          // keeper only: the CTA's next tile (i + 1 at the top of iteration i)
    if (keeper && t < n_tiles) {
        const Tile d0 = tiles[t];
        s.tdesc[0] = d0;
        issue_lean_loads<PROP, CULL, WITH_TRS>(R, d0, s.st[0], &s.bar[0]);
    }
    __syncthreads();      // barriers initialised, planes and the first descriptor staged
    if (keeper && t < n_tiles) {
        // Tile hand-out: a CTA starts on tile blockIdx.x and then takes the tiles the grid has not started yet in ticket order.
        // The ticket counter is never reset: every launch draws exactly n_tiles tickets, and the host passes the running base.
        // (behind the barrier: only this thread's warp waits for the atomic)
        k_next = ticket ? gridDim.x + (atomicAdd(ticket, 1u) - ticket_base) : t + gridDim.x;
        if (k_next < n_tiles) cp_async_tile_desc(&s.tdesc[1], tiles + k_next);
    }
    uint32_t n_gt_total = 0, n_vv_total = 0;
    uint32_t slot = 0;                  // it % 3
    for (uint32_t it = 0; t < n_tiles; ++it) {
        const uint32_t sidx = it & 1u;
        const uint32_t pp = PIPE ? sidx : 0u;        // which copy of the per-tile scratch
        const uint32_t slot1 = slot == 2u ? 0u : slot + 1u;
        LeanStage<WITH_TRS> &S = s.st[sidx];
        if constexpr (PIPE) {
            // the tile has landed -- or the bookkeeping thread has signalled that there is none; either way what it wrote before
            // (next tile index, the tile's descriptor) is visible behind this wait
            mbar_wait(&s.bar[sidx], (it >> 1) & 1u);
            if (it > 0u) { t = s.next_tile[sidx ^ 1u]; if (t >= n_tiles) break; }
        }
        const uint2 tb = *reinterpret_cast<const uint2 *>(&s.tdesc[slot]);     // base | n_rows, n_levels
        const uint32_t tile_base = tb.x, tile_rows = tb.y & 0xFFFFu, tile_levels = tb.y >> 16;
        const uint32_t off = tile_base & 15u;
        const uint32_t li = off + lr;                 // index into the staged window
        const bool active = lr < tile_rows;
        const uint32_t row = tile_base + lr;
        // columns that are not staged: plain coalesced loads issued above the wait for the tile.  Transform (MINB > 4) is consumed
        // right behind the tile's opening barrier, the bounds only after the hierarchy walk
        float4 tA = make_float4(0, 0, 0, 1), tB = make_float4(0, 0, 0, 1); float2 tC = make_float2(1, 1);
        if (PROP && !WITH_TRS && active) { tA = R.trsA[row]; tB = R.trsB[row]; tC = R.trsC[row]; }
        float4 bA = make_float4(0, 0, 0, 0); float2 bB = make_float2(0, 0);
        if (CULL && active) { bA = R.bndA[row]; bB = R.bndB[row]; }
        if constexpr (!PIPE) mbar_wait(&s.bar[sidx], (it >> 1) & 1u);
        const uint32_t f = active ? S.flags[li] : 0u;
        const uint32_t st8 = active ? S.state[li] : 0u;

        // The bookkeeping thread prefetches the NEXT tile a whole walk ahead of its use: the other stage was last read by the
        // previous tile's bulk store (issued just before, so this thread may wait here -- its warp has nothing to do until the
        // levels above its rows are walked), and the next tile's descriptor was fetched while the previous tile was culled.
        auto prefetch_next = [&]() {
            const uint32_t tn = k_next;
            s.next_tile[sidx] = tn;      // read by everybody behind the tile's closing barrier (PIPE: behind the next stage's TMA barrier)
            if (tn < n_tiles) {
                asm volatile("cp.async.wait_all;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                const Tile dn = s.tdesc[slot1];
                issue_lean_loads<PROP, CULL, WITH_TRS>(R, dn, s.st[sidx ^ 1u], &s.bar[sidx ^ 1u]);
                k_next = ticket ? gridDim.x + (atomicAdd(ticket, 1u) - ticket_base) : tn + gridDim.x;   // consumed after the walk
            } else if (PIPE) {
                mbar_arrive_cta(&s.bar[sidx ^ 1u]);      // no more tiles: complete the phase the CTA's warps will wait on
            }
        };
        if (!PROP && keeper) prefetch_next();
        bool visited = false, changed = false;
        if (PROP) {
            const uint32_t topo = active ? S.topo[li] : T_DETACHED;
            const uint32_t depth = (topo >> 9) & 0x1FFu, plocal = topo & 0x1FFu;
            const bool tchanged = f & F_TCHANGED;
            const bool has_children = topo & T_HAS_CHILDREN;
            bool dirty = tchanged;
            bool climbed = false;      // s.dirty[] holds this tile's TransformTreeChanged bits
            bool must_climb = false;
            if (static_opt && R.dirty == nullptr && tile_levels > 1) {
                if constexpr (PIPE) {
                    // every warp answers for the whole tile from the staged columns: 8 rows per lane, no CTA-wide vote
                    const uint32_t r0 = (lr & 31u) * 8u;
                    bool mine = false;
#pragma unroll
                    for (uint32_t j = 0; j < 8u; ++j)
                        if (r0 + j < tile_rows) mine |= (S.flags[off + r0 + j] & F_TCHANGED) && (((S.topo[off + r0 + j] >> 9) & 0x1FFu) > 0u);
                    must_climb = __any_sync(0xFFFFFFFFu, mine);
                } else {
                    must_climb = __syncthreads_or(tchanged && depth > 0);
                }
            }
            if (static_opt && R.dirty != nullptr) {
                dirty = active && R.dirty[row];
            } else if (must_climb) {
                climbed = true;
                // only when a non-root row of the tile changed does anything have to climb: otherwise every row's
                // TransformTreeChanged bit equals its own Changed<Transform> bit (one barrier instead of two + a climb)
                s.parent[lr] = (uint16_t)((depth > 0) ? plocal : 0xFFFFu);
                s.dirty[lr] = 0;
                __syncthreads();
                if (active && tchanged) {
                    uint32_t c = lr;
                    while (!s.dirty[c]) {
                        s.dirty[c] = 1;
                        const uint32_t p = s.parent[c];
                        if (p == 0xFFFFu) break;
                        c = p;
                    }
                }
                __syncthreads();
                dirty = s.dirty[lr];
            }
            if (keeper) prefetch_next();      // behind the tile's opening barrier(s): the walk's first warp never waits for it
            const uint32_t my_level = (active && !(topo & T_DETACHED)) ? depth : 0xFFFFFFFFu;
            if (active && (topo & T_DETACHED) && has_children) s.pst[pp][lr] = 0;
            // ---- the tile's TOP LEVELS in registers (tiles whose first K >= 2 depth levels sit among the first 32 rows: a BFS-ordered
            // tree).  The rows of those levels form a serial chain of K matrix products that every other row of the tile waits for.
            // Level by level through shared memory that chain costs a store / __syncwarp / load round trip and a pass through the
            // level loop per level, all in ONE warp.  Here that warp keeps every row's GlobalTransform in registers and a child fetches
            // its parent's matrix (and visited / changed bits) with warp shuffles: 13 SHFL + the product + set_if_neq per level,
            // nothing goes through shared memory until the lanes store their own rows at the end.
            uint32_t top_k = 0;
            unsigned long long lvl_warps = 0ull; uint32_t wsm = 0;
            if (tile_levels > 1u) {
                wsm = s.tdesc[slot].warp_sync_mask; lvl_warps = s.tdesc[slot].lvl_warps;
                if (lvl_warps != 0ull && (probe & 4u) == 0u) { top_k = s.tdesc[slot].top_levels; if (top_k < 2u) top_k = 0u; }
            }
            if constexpr (WITH_TRS) { tA = S.trsA[li]; tB = S.trsB[li]; tC = S.trsC[li]; }
            const Aff l = affine_from_trs(tA, tB, tC);
            if (top_k && lr < 32u) {
                Aff G; G.r0 = S.gt0[li]; G.r1 = S.gt1[li]; G.r2 = S.gt2[li];      // last frame's value (set_if_neq keeps it when equal)
                bool vis = false, chg = false;
                if (my_level == 0u) {
                    if (topo & T_ROOT) {
                        vis = has_children ? (!static_opt || dirty) : tchanged;
                        chg = vis;
                        if (vis) G = l;
                    } else {
                        const uint32_t pr = R.parent[row];
                        const uint32_t ps = R.state[pr];
                        vis = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                        if (vis) {
                            Aff n;
                            n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                            chg = row_neq(n.r0, G.r0) | row_neq(n.r1, G.r1) | row_neq(n.r2, G.r2);
                            if (chg) G = n;
                        }
                    }
                }
                for (uint32_t d = 1; d < top_k; ++d) {
                    // (a detached row publishes vis = 0, like its pst byte; lanes whose parent is not in this warp read garbage and ignore it)
                    const uint32_t pv = __shfl_sync(0xFFFFFFFFu, (vis ? 1u : 0u) | (chg ? 2u : 0u), plocal);
                    Aff P;
                    P.r0.x = __shfl_sync(0xFFFFFFFFu, G.r0.x, plocal); P.r0.y = __shfl_sync(0xFFFFFFFFu, G.r0.y, plocal);
                    P.r0.z = __shfl_sync(0xFFFFFFFFu, G.r0.z, plocal); P.r0.w = __shfl_sync(0xFFFFFFFFu, G.r0.w, plocal);
                    P.r1.x = __shfl_sync(0xFFFFFFFFu, G.r1.x, plocal); P.r1.y = __shfl_sync(0xFFFFFFFFu, G.r1.y, plocal);
                    P.r1.z = __shfl_sync(0xFFFFFFFFu, G.r1.z, plocal); P.r1.w = __shfl_sync(0xFFFFFFFFu, G.r1.w, plocal);
                    P.r2.x = __shfl_sync(0xFFFFFFFFu, G.r2.x, plocal); P.r2.y = __shfl_sync(0xFFFFFFFFu, G.r2.y, plocal);
                    P.r2.z = __shfl_sync(0xFFFFFFFFu, G.r2.z, plocal); P.r2.w = __shfl_sync(0xFFFFFFFFu, G.r2.w, plocal);
                    if (my_level == d) {
                        vis = (pv & 1u) && !(static_opt && !dirty && !(pv & 2u));
                        if (vis) {
                            Aff n;
                            n.r0 = affine_mul_row(P.r0, l); n.r1 = affine_mul_row(P.r1, l); n.r2 = affine_mul_row(P.r2, l);
                            chg = row_neq(n.r0, G.r0) | row_neq(n.r1, G.r1) | row_neq(n.r2, G.r2);   // set_if_neq
                            if (chg) G = n;
                        }
                    }
                }
                if (my_level < top_k) {
                    visited = vis; changed = chg;
                    if (chg) { S.gt0[li] = G.r0; S.gt1[li] = G.r1; S.gt2[li] = G.r2; }
                    if (has_children) s.pst[pp][lr] = (uint8_t)((vis ? 1u : 0u) | (chg ? 2u : 0u));
                }
            }
            if (my_level == 0 && !top_k) {
                Aff n = l;
                if (topo & T_ROOT) {
                    visited = has_children ? (!static_opt || dirty) : tchanged;
                    changed = visited;
                } else {
                    const uint32_t pr = R.parent[row];
                    const uint32_t ps = R.state[pr];
                    visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                    if (visited) {
                        n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                        changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);
                    }
                }
                if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                if (has_children) s.pst[pp][lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            }
            // one level of the walk for this thread's row: the parent's rows are the tile's own (in-place) GlobalTransform entries
            auto walk_row = [&]() {
                const uint32_t pst = s.pst[pp][plocal];
                const uint32_t pi = off + plocal;
                visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                if (visited) {
                    Aff n;
                    n.r0 = affine_mul_row(S.gt0[pi], l); n.r1 = affine_mul_row(S.gt1[pi], l); n.r2 = affine_mul_row(S.gt2[pi], l);
                    changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);   // set_if_neq
                    if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                }
                if (has_children) s.pst[pp][lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            };
            if (tile_levels > 1u) {
                if (lvl_warps != 0ull) {
                    // per-warp level schedule through named barriers (see kernel 1b)
                    const uint32_t lmask = __reduce_or_sync(0xFFFFFFFFu, active ? (1u << (depth & 15u)) : 0u);
                    uint32_t need = (lmask | (lmask << 1)) & ((1u << tile_levels) - 2u);
                    if (top_k) need &= ~((1u << top_k) - 2u);       // levels 1 .. K-1 were walked in registers above
                    while (need) {
                        const uint32_t lvl = (uint32_t)__ffs((int)need) - 1u;
                        need &= need - 1u;
                        const bool consumer = (lmask >> lvl) & 1u;
                        if ((wsm >> lvl) & 1u) {       // every edge into this level stays inside a warp
                            if (!consumer) continue;
                            if (!((probe & 3u) == 1u || ((probe & 3u) == 2u && lvl < 5u))) __syncwarp();
                        } else if ((probe & 3u) == 1u || ((probe & 3u) == 2u && lvl < 5u)) {     // timing probe: no hand-over at all (races; wrong results)
                            if (!consumer) continue;
                        } else {
                            const uint32_t cnt = ((uint32_t)(lvl_warps >> (4u * lvl)) & 15u) * 32u;
                            if (!consumer) {
                                asm volatile("fence.acq_rel.cta;" ::: "memory");
                                // (4 CTAs per SM may own 16 hardware barriers each: a register id costs nothing there)
                                if constexpr (PIPE) asm volatile("bar.arrive %0, %1;" ::"r"(lvl + 8u * sidx), "r"(cnt) : "memory");
                                else if constexpr (MINB <= 4) asm volatile("bar.arrive %0, %1;" ::"r"(lvl), "r"(cnt) : "memory");
                                else named_bar_arrive(lvl, cnt);
                                continue;
                            }
                            if constexpr (PIPE) asm volatile("bar.sync %0, %1;" ::"r"(lvl + 8u * sidx), "r"(cnt) : "memory");
                            else if constexpr (MINB <= 4) asm volatile("bar.sync %0, %1;" ::"r"(lvl), "r"(cnt) : "memory");
                            else named_bar_sync(lvl, cnt);
                        }
                        if (my_level == lvl) walk_row();
                    }
                } else {
                    for (uint32_t lvl = 1; lvl < tile_levels; ++lvl) {
                        if (lvl < 32u && ((wsm >> lvl) & 1u)) __syncwarp(); else __syncthreads();
                        if (my_level == lvl) walk_row();
                    }
                }
            }
            if (active && tchanged) R.flags[row] = (uint8_t)(f & ~F_TCHANGED);
        }
        // the descriptor of the tile after next: the ticket drawn at the top of this tile is back by now
        if (keeper && k_next < n_tiles) cp_async_tile_desc(&s.tdesc[slot == 0u ? 2u : slot - 1u], tiles + k_next);
        uint32_t out = st8 & (S_VV | S_HAS_CLASS);
        if (PROP) out |= (changed ? S_GT_CHANGED : 0u) | (visited ? S_VISITED : 0u);
        else out |= st8 & (S_GT_CHANGED | S_VISITED);

        bool vv_changed = false;
        if (CULL) {
            Aff g; g.r0 = S.gt0[li]; g.r1 = S.gt1[li]; g.r2 = S.gt2[li];   // own row: written by this thread or untouched
            const bool in_query = active && !(f & F_NO_CPU_CULL);
            const bool base = in_query && (f & F_INHERITED);
            const uint32_t prev = st8 & 1u;
            const uint32_t lane = lr & 31u;
            const bool has_aabb = f & F_AABB;
            const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
            float cx, cy, cz, radius;
            const float hx = bA.w, hy = bB.x, hz = bB.y;
            if (has_aabb) {
                cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
                cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
                cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
                const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
                const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
                const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
                radius = sqrtf((vx * vx + vy * vy) + vz * vz);
            } else {
                const bool from_gt = f & F_SPHERE_GT;
                cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
                radius = bA.w;
            }
            unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
            if (!SIMPLE && active) {
                if (R.layers != nullptr) elayers = R.layers[row];
                if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
                if (R.rank != nullptr) rnk = R.rank[row];
            }
            // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
            const uint32_t rejmask = (probe & 8u) ? warp_view_reject_sphere(s.vplanes, s.vlen, cvw.n_views, base && do_test, base && !do_test, cx, cy, cz, radius)
                                                 : warp_view_reject_lean(s.vplanes, cvw.n_views, base && do_test, base && !do_test, cx, cy, cz, radius);
            uint32_t todo = v_on & ~(rejmask & ~v_nofr);     // a NoCpuCulling camera lists without frustum tests: never rejected
            bool any = false;
            uint32_t my_ballot = 0;
            while (todo) {
                const uint32_t v = (uint32_t)__ffs((int)todo) - 1u;
                todo &= todo - 1u;
                bool vis = base;
                if (!SIMPLE) {
                    vis = vis && layers_intersect(R, cvw, row, v, elayers);
                    if ((f & F_RANGE) && R.range != nullptr) {
                        const int32_t ri = cvw.range_index[v];
                        vis = vis && ri >= 0 && ((erange >> ri) & 1u);
                    }
                }
                if (do_test && !((v_nofr >> v) & 1u)) {
                    const float4 *pl = s.vplanes + v * 5u;
                    float d[5];
                    bool out_s = false;
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        d[k] = plane_dot_point(pl[k], cx, cy, cz);
                        out_s |= (d[k] + radius <= 0.0f);
                    }
                    vis = vis && !out_s;
                    if (vis && has_aabb) {
                        bool out_o = false;
#pragma unroll
                        for (int k = 0; k < 5; ++k) {
                            const float4 n = pl[k];
                            const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                            const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                            const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                            const float rr = (dx * hx + dy * hy) + dz * hz;
                            out_o |= (d[k] + rr <= 0.0f);
                        }
                        vis = !out_o;
                    }
                }
                any |= vis;
                const bool listed = vis && (st8 & S_HAS_CLASS);
                if (SIMPLE || R.rank == nullptr) {
                    const uint32_t b = __ballot_sync(0xFFFFFFFFu, listed);
                    if (lane == v) my_ballot = b;
                } else if (listed) {
                    uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
                    uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
                    atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                    atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
                }
            }
            if (my_ballot) {
                uint32_t *mask = vb.mask + (size_t)lane * vb.words_stride;
                uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride;
                const uint32_t row0 = row - lane, w0 = row0 >> 5, sh = row0 & 31u;
                const uint32_t lo = my_ballot << sh, hi = sh ? (my_ballot >> (32u - sh)) : 0u;
                if (lo) { atomicOr(mask + w0, lo); atomicAdd(cc + (w0 / kChunkWords), __popc(lo)); }
                if (hi) { atomicOr(mask + w0 + 1, hi); atomicAdd(cc + ((w0 + 1) / kChunkWords), __popc(hi)); }
            }
            if (in_query) {
                out = (out & ~S_VV) | (any ? (1u | (prev << 1)) : 0u);
                vv_changed = (any ? 1u : 0u) != prev;
                if (vv_changed) out |= S_VV_CHANGED;
            }
        } else {
            out |= st8 & S_VV_CHANGED;
        }
        if (active && out != st8) R.state[row] = (uint8_t)out;
        // a light row publishes what assign_objects_to_clusters needs of it (GlobalTransform::translation,
        // ViewVisibility::get) so that the cluster kernels never touch the row arrays again
        if (CULL && R.light_snap != nullptr && (f & F_SPHERE_GT) && active) {
            const uint32_t ord = R.light_ord[row];     // 0xFFFFFFFF: a sphere-from-GT row that is not a current light
            if (ord < R.n_lights) R.light_snap[ord] = make_float4(S.gt0[li].w, S.gt1[li].w, S.gt2[li].w, (out & 1u) ? 1.0f : 0.0f);
        }

        // end of tile: everybody is done with this stage; count changes; write the tile's matrices back
        n_gt_total += (PROP && changed) ? 1u : 0u;      // per-thread tallies, reduced once at the end of the kernel
        n_vv_total += vv_changed ? 1u : 0u;
        int any_gt;
        if constexpr (PIPE) {
            // this warp is through with the stage: say so and move on; only the bookkeeping thread waits for the other warps
            if (__any_sync(0xFFFFFFFFu, changed) && (lr & 31u) == 0u) s.anyflag[sidx] = 1u;
            __syncwarp();
            if ((lr & 31u) == 0u) mbar_arrive_cta(&s.done[sidx]);
            any_gt = 0;
            if (keeper) {
                mbar_wait_guarded(&s.done[sidx], (it >> 1) & 1u);
                any_gt = (int)s.anyflag[sidx];
                s.anyflag[sidx] = 0u;       // the next writers (two tiles on) start behind the load this thread issues after this
            }
        } else {
            any_gt = __syncthreads_or(PROP && changed);
            t = s.next_tile[sidx];
        }
        if (keeper && PROP && any_gt) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic smem writes -> async proxy
            const uint32_t bytes = tile_rows * 16u;
            bulk_s2g(R.gt0 + tile_base, S.gt0 + off, bytes); bulk_s2g(R.gt1 + tile_base, S.gt1 + off, bytes);
            bulk_s2g(R.gt2 + tile_base, S.gt2 + off, bytes);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        slot = slot1;
    }
    if (keeper) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    // block-reduce the per-thread tallies (warp shuffle, then one shared-memory atomic per warp)
    __shared__ uint32_t s_cnt[2];
    if (lr < 2) s_cnt[lr] = 0;
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { n_gt_total += __shfl_xor_sync(0xFFFFFFFFu, n_gt_total, o); n_vv_total += __shfl_xor_sync(0xFFFFFFFFu, n_vv_total, o); }
    if ((lr & 31u) == 0) { if (n_gt_total) atomicAdd(&s_cnt[0], n_gt_total); if (n_vv_total) atomicAdd(&s_cnt[1], n_vv_total); }
    __syncthreads();
    if (lr == 0) {
        if (s_cnt[0]) atomicAdd(&stats->changed[parity][0], s_cnt[0]);
        if (s_cnt[1]) atomicAdd(&stats->changed[parity][1], s_cnt[1]);
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 1f (B200VIS_TILE_KERNEL=flow): the TMA-staged pass WITHOUT a CTA-wide barrier between tiles, per-warp level hand-overs
// through named barriers, GlobalTransforms stored straight from registers.  Parity-clean, measured slower than kernel 1b
// (DESIGN.md section 7): kept selectable as the record of that experiment.
// ------------------------------------------------------------------------------------------
template <bool PROP, bool CULL, bool SIMPLE>
__global__ void __launch_bounds__(kTileRows, 4)
k_propagate_cull_flow(Rows R, const Tile *__restrict__ tiles, uint32_t n_tiles, const __grid_constant__ CullViews cvw,
                     VisibleBufs vb, DevStats *__restrict__ stats, uint32_t static_opt, uint32_t parity,
                     uint32_t *__restrict__ /*ticket*/, uint32_t /*ticket_base*/) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    TmaSmem &s = *reinterpret_cast<TmaSmem *>(smem_raw);
    const uint32_t lr = threadIdx.x;
    if (lr == 0) {
        mbar_init(&s.bar[0], 1); mbar_init(&s.bar[1], 1);
        mbar_init(&s.walked[0], kTileRows / 32); mbar_init(&s.walked[1], kTileRows / 32);
        s.climb[0] = 0; s.climb[1] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // launched with programmatic stream serialization: everything above overlapped the previous kernel's tail
    TT(0);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    TT(1);
    // ---- Tile FLOW --------------------------------------------------------------------------------------------------------
    // A tile's hierarchy walk is a chain of its levels; the cull that follows is wide.  There is NO CTA-wide barrier between
    // tiles: a warp that has walked its rows of tile k takes them into registers, looks at tile k+1's change flags
    // (mark_dirty_trees: does anything have to climb?), arrives on walked[stage] and culls; whoever is done culling goes on to
    // tile k+1 and starts its walk as soon as walked[stage of k] completes -- that is, when the LAST warp has left tile k's
    // walk, while those last (leaf-level) warps are still culling.  So the chain of tile k+1 runs under the cull of tile k, in
    // the same CTA, and the SM always has wide work to issue.  Hand-overs:
    //   full[s]    TMA -> all       tile landed in stage s                       (loads issued one tile ahead by thread 0)
    //   walked[s]  8 warps -> all   stage s free, pst/parent/dirty free, climb[s ^ 1] final
    //   named barriers 1..7 (even tiles) / 8..14 (odd tiles): the level hand-overs inside a walk (Tile::lvl_warps)
    // A warp is never more than one tile ahead of another (it needs walked[] of the tile before), which is what makes two
    // stages, one pst array and two barrier-id sets enough.
    uint32_t t = blockIdx.x;
    if (lr == 0 && t < n_tiles) issue_tile_loads<PROP, CULL>(R, tiles[t], s.st[0], &s.bar[0]);
    uint32_t n_gt_total = 0, n_vv_total = 0;
    const bool scan_flags = PROP && static_opt && R.dirty == nullptr;     // in-tile mark_dirty_trees (single-pass plans)
    for (uint32_t it = 0; t < n_tiles; t += gridDim.x, ++it) {
        const uint32_t sidx = it & 1u;
        const Tile tile = tiles[t];
        const uint32_t tn = t + gridDim.x;
        const bool has_next = tn < n_tiles;
        // the previous tile (other stage) is walked by everybody: its stage, the pst/parent/dirty arrays and this tile's climb
        // flag are ours now
        if (it > 0) mbar_wait_guarded(&s.walked[sidx ^ 1u], ((it - 1u) >> 1) & 1u);
        if (lr == 0 && has_next) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the stage's old generic accesses -> async proxy
            issue_tile_loads<PROP, CULL>(R, tiles[tn], s.st[sidx ^ 1u], &s.bar[sidx ^ 1u]);
        }
        mbar_wait_guarded(&s.bar[sidx], (it >> 1) & 1u);
        if (it == 1) { TT(2); }
        TileStage &S = s.st[sidx];
        const uint32_t off = tile.base & 15u;
        const uint32_t li = off + lr;                 // index into the staged window
        const bool active = lr < tile.n_rows;
        const uint32_t row = tile.base + lr;
        const uint32_t f = active ? S.flags[li] : 0u;
        const uint32_t st8 = active ? S.state[li] : 0u;
        // bounds are only needed after the hierarchy walk: plain coalesced loads issued now, consumed in the cull
        // (keeping them out of the staged window lets a fourth CTA fit in shared memory)
        float4 bA = make_float4(0, 0, 0, 0); float2 bB = make_float2(0, 0);
        if (CULL && active) { bA = R.bndA[row]; bB = R.bndB[row]; }
        const uint32_t topo = (PROP && active) ? S.topo[li] : T_DETACHED;
        const uint32_t depth = (topo >> 9) & 0x1FFu, plocal = topo & 0x1FFu;
        const bool tchanged = PROP && (f & F_TCHANGED);
        // mark_dirty_trees: only when a non-root row of the tile changed does anything have to climb; otherwise every row's
        // TransformTreeChanged bit equals its own Changed<Transform> bit.  The first tile asks the CTA; later tiles were looked
        // at by every warp on its way out of the previous walk.
        bool climb = false;
        if (scan_flags && tile.n_levels > 1) climb = (it == 0) ? (__syncthreads_or(tchanged && depth > 0) != 0) : (s.climb[sidx] == it);

        bool visited = false, changed = false;
        if (PROP) {
            const bool has_children = topo & T_HAS_CHILDREN;
            bool dirty = tchanged;
            if (static_opt && R.dirty != nullptr) {
                dirty = active && R.dirty[row];
            } else if (climb) {
                s.parent[lr] = (uint16_t)((depth > 0) ? plocal : 0xFFFFu);
                s.dirty[lr] = 0;
                __syncthreads();
                if (active && tchanged) {
                    uint32_t c = lr;
                    while (!s.dirty[c]) {
                        s.dirty[c] = 1;
                        const uint32_t p = s.parent[c];
                        if (p == 0xFFFFu) break;
                        c = p;
                    }
                }
                __syncthreads();
                dirty = s.dirty[lr];
            }
            if (it == 1) { TT(3); }    // dirty phase done
            const Aff l = affine_from_trs(S.trsA[li], S.trsB[li], S.trsC[li]);
            const uint32_t my_level = (active && !(topo & T_DETACHED)) ? depth : 0xFFFFFFFFu;
            if (active && (topo & T_DETACHED) && has_children) s.pst[lr] = 0;
            // set_if_neq, in place in the staged tile (where a row's in-tile children read it)
            auto commit = [&](const Aff &n) {
                changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);
                if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
            };
            if (my_level == 0) {
                if (topo & T_ROOT) {
                    visited = has_children ? (!static_opt || dirty) : tchanged;
                    changed = visited;
                    // roots are written without a compare (systems.rs: `*gt = GlobalTransform::from(*t)`)
                    if (changed) { S.gt0[li] = l.r0; S.gt1[li] = l.r1; S.gt2[li] = l.r2; }
                } else {
                    const uint32_t pr = R.parent[row];
                    const uint32_t ps = R.state[pr];
                    visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                    if (visited) {
                        Aff n;
                        n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                        commit(n);
                    }
                }
                if (has_children) s.pst[lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            }
            if (it == 1) { TT(4); }    // local affine + level 0 done
            // one level of the walk for this thread's row: the parent's rows are the tile's own (in-place) GlobalTransform entries
            auto walk_row = [&]() {
                const uint32_t pst = s.pst[plocal];
                const uint32_t pi = off + plocal;
                visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                if (visited) {
                    Aff n;
                    n.r0 = affine_mul_row(S.gt0[pi], l); n.r1 = affine_mul_row(S.gt1[pi], l); n.r2 = affine_mul_row(S.gt2[pi], l);
                    commit(n);
                }
                if (has_children) s.pst[lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
            };
            if (tile.lvl_warps != 0ull) {
                // Per-warp level schedule (2..8 levels).  A warp only takes part in the hand-over of the levels its own rows
                // produce (level l-1) or consume (level l), through hardware named barrier l with exactly the warps the planner
                // counted (Tile::lvl_warps): consumers bar.sync, pure producers bar.arrive and go on.  The warps that hold a
                // tree's upper levels are thus culling while the chain is still running down the lower ones, a leaf warp waits
                // once instead of once per level, and nobody pays the loop for levels that are not theirs.
                // (a detached row takes no part in the walk but publishes pst = 0 for its children: it counts as a level-0 row)
                const uint32_t lmask = __reduce_or_sync(0xFFFFFFFFu, active ? (1u << (depth & 15u)) : 0u);
                uint32_t need = (lmask | (lmask << 1)) & ((1u << tile.n_levels) - 2u);
                while (need) {
                    const uint32_t lvl = (uint32_t)__ffs((int)need) - 1u;
                    need &= need - 1u;
                    const bool consumer = (lmask >> lvl) & 1u;
                    if ((tile.warp_sync_mask >> lvl) & 1u) {       // every edge into this level stays inside a warp
                        if (!consumer) continue;
                        __syncwarp();
                    } else {
                        const uint32_t cnt = ((uint32_t)(tile.lvl_warps >> (4u * lvl)) & 15u) * 32u;
                        const uint32_t id = lvl + sidx * 7u;        // levels 1..7; two id sets: a warp may be one tile ahead
                        if (!consumer) {
                            __threadfence_block();
                            asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(cnt) : "memory");
                            continue;
                        }
                        asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(cnt) : "memory");
                    }
                    if (my_level == lvl) walk_row();
                }
            } else {
                for (uint32_t lvl = 1; lvl < tile.n_levels; ++lvl) {
                    if (lvl < 32u && ((tile.warp_sync_mask >> lvl) & 1u)) __syncwarp(); else __syncthreads();
                    if (my_level == lvl) walk_row();
                    if (it == 1 && lvl <= 7) { TT(4 + lvl); }   // thread 0 after the level's barrier and (for level-lvl rows) work
                }
            }
            if (active && tchanged) R.flags[row] = (uint8_t)(f & ~F_TCHANGED);
        }
        if (it == 1) { TT(12); }   // walk done
        uint32_t out = st8 & (S_VV | S_HAS_CLASS);
        if (PROP) out |= (changed ? S_GT_CHANGED : 0u) | (visited ? S_VISITED : 0u);
        else out |= st8 & (S_GT_CHANGED | S_VISITED);

        // on the way out of the walk: the next tile's change flags (it landed while this one was walked) ...
        if (scan_flags && has_next) {
            const Tile nt = tiles[tn];
            if (nt.n_levels > 1) {
                mbar_wait_guarded(&s.bar[sidx ^ 1u], ((it + 1u) >> 1) & 1u);
                const TileStage &N = s.st[sidx ^ 1u];
                const uint32_t nli = (nt.base & 15u) + lr;
                const bool hit = lr < nt.n_rows && (N.flags[nli] & F_TCHANGED) && ((N.topo[nli] >> 9) & 0x1FFu) != 0u && !(N.topo[nli] & T_DETACHED);
                if (__any_sync(0xFFFFFFFFu, hit) && (lr & 31u) == 0) s.climb[sidx ^ 1u] = it + 1u;     // stamped with the tile's iteration: never cleared
            }
        }
        // ... then the own row -- written by this thread or untouched -- into registers (a changed matrix goes to HBM straight
        // from them: three coalesced 512-byte stores per warp), and walked[stage]: this warp is done with the staged tile
        Aff g; g.r0 = S.gt0[li]; g.r1 = S.gt1[li]; g.r2 = S.gt2[li];
        if (PROP && changed) { R.gt0[row] = g.r0; R.gt1[row] = g.r1; R.gt2[row] = g.r2; }
        __syncwarp();
        if ((lr & 31u) == 0) mbar_arrive_cta(&s.walked[sidx]);
        bool vv_changed = false;
        if (CULL) {
            const bool in_query = active && !(f & F_NO_CPU_CULL);
            const bool base = in_query && (f & F_INHERITED);
            const bool rej_base = base;
            const uint32_t prev = st8 & 1u;
            const uint32_t lane = lr & 31u;
            const bool has_aabb = f & F_AABB;
            const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
            float cx, cy, cz, radius;
            const float hx = bA.w, hy = bB.x, hz = bB.y;
            if (has_aabb) {
                cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
                cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
                cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
                const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
                const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
                const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
                radius = sqrtf((vx * vx + vy * vy) + vz * vz);
            } else {
                const bool from_gt = f & F_SPHERE_GT;
                cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
                radius = bA.w;
            }
            unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
            if (!SIMPLE && active) {
                if (R.layers != nullptr) elayers = R.layers[row];
                if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
                if (R.rank != nullptr) rnk = R.rank[row];
            }
            // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
            const uint32_t rejmask = warp_view_reject(cvw, rej_base && do_test, rej_base && !do_test, cx, cy, cz, radius);
            bool any = false;
            uint32_t my_ballot = 0;
#pragma unroll
            for (uint32_t v = 0; v < kMaxViews; ++v) {
                if (v >= cvw.n_views) break;
                const uint32_t von = cvw.on[v];
                if (!(von & 1u)) continue;
                if (SIMPLE && !(von & 4u)) continue;   // bit2: the view includes the default layer
                if (((rejmask >> v) & 1u) && !(von & 2u)) continue;         // every row of this warp is outside this view's frustum
                bool vis = base;
                if (!SIMPLE) {
                    vis = vis && layers_intersect(R, cvw, row, v, elayers);
                    if ((f & F_RANGE) && R.range != nullptr) {
                        const int32_t ri = cvw.range_index[v];
                        vis = vis && ri >= 0 && ((erange >> ri) & 1u);
                    }
                }
                if (do_test && !(von & 2u)) {
                    const float d0 = plane_dot_point(cvw.planes[v][0], cx, cy, cz), d1 = plane_dot_point(cvw.planes[v][1], cx, cy, cz);
                    const float d2 = plane_dot_point(cvw.planes[v][2], cx, cy, cz), d3 = plane_dot_point(cvw.planes[v][3], cx, cy, cz);
                    const float d4 = plane_dot_point(cvw.planes[v][4], cx, cy, cz);
                    const bool out_s = (d0 + radius <= 0.0f) | (d1 + radius <= 0.0f) | (d2 + radius <= 0.0f) |
                                       (d3 + radius <= 0.0f) | (d4 + radius <= 0.0f);
                    vis = vis && !out_s;
                    if (vis && has_aabb) {
                        const float d[5] = {d0, d1, d2, d3, d4};
                        bool out_o = false;
#pragma unroll
                        for (int k = 0; k < 5; ++k) {
                            const float4 n = cvw.planes[v][k];
                            const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                            const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                            const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                            const float rr = (dx * hx + dy * hy) + dz * hz;
                            out_o |= (d[k] + rr <= 0.0f);
                        }
                        vis = !out_o;
                    }
                }
                any |= vis;
                const bool listed = vis && (st8 & S_HAS_CLASS);
                if (SIMPLE || R.rank == nullptr) {
                    const uint32_t b = __ballot_sync(0xFFFFFFFFu, listed);
                    if (lane == v) my_ballot = b;
                } else if (listed) {
                    uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
                    uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
                    atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                    atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
                }
            }
            if (my_ballot) {
                uint32_t *mask = vb.mask + (size_t)lane * vb.words_stride;
                uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride;
                const uint32_t row0 = row - lane, w0 = row0 >> 5, sh = row0 & 31u;
                const uint32_t lo = my_ballot << sh, hi = sh ? (my_ballot >> (32u - sh)) : 0u;
                if (lo) { atomicOr(mask + w0, lo); atomicAdd(cc + (w0 / kChunkWords), __popc(lo)); }
                if (hi) { atomicOr(mask + w0 + 1, hi); atomicAdd(cc + ((w0 + 1) / kChunkWords), __popc(hi)); }
            }
            if (in_query) {
                out = (out & ~S_VV) | (any ? (1u | (prev << 1)) : 0u);
                vv_changed = (any ? 1u : 0u) != prev;
                if (vv_changed) out |= S_VV_CHANGED;
            }
            // a light row publishes what assign_objects_to_clusters needs of it (GlobalTransform::translation,
            // ViewVisibility::get) so that the cluster kernels never touch the row arrays again
            if (R.light_snap != nullptr && (f & F_SPHERE_GT) && active) {
                const uint32_t ord = R.light_ord[row];     // 0xFFFFFFFF: a sphere-from-GT row that is not a current light
                if (ord < R.n_lights) R.light_snap[ord] = make_float4(g.r0.w, g.r1.w, g.r2.w, (out & 1u) ? 1.0f : 0.0f);
            }
        } else {
            out |= st8 & S_VV_CHANGED;
        }
        if (active && out != st8) R.state[row] = (uint8_t)out;
        n_gt_total += (PROP && changed) ? 1u : 0u;      // per-thread tallies, reduced once at the end of the kernel
        n_vv_total += vv_changed ? 1u : 0u;
        if (it == 1) { TT(13); }   // cull done: no barrier here -- the warp goes on to the next tile's rendezvous
    }
    TT(14);
    // block-reduce the per-thread tallies (warp shuffle, then one shared-memory atomic per warp)
    __shared__ uint32_t s_cnt[2];
    if (lr < 2) s_cnt[lr] = 0;
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { n_gt_total += __shfl_xor_sync(0xFFFFFFFFu, n_gt_total, o); n_vv_total += __shfl_xor_sync(0xFFFFFFFFu, n_vv_total, o); }
    if ((lr & 31u) == 0) { if (n_gt_total) atomicAdd(&s_cnt[0], n_gt_total); if (n_vv_total) atomicAdd(&s_cnt[1], n_vv_total); }
    __syncthreads();
    if (lr == 0) {
        if (s_cnt[0]) atomicAdd(&stats->changed[parity][0], s_cnt[0]);
        if (s_cnt[1]) atomicAdd(&stats->changed[parity][1], s_cnt[1]);
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 1s: the TMA-staged CTA-per-tile pass with a SCOUT warp.
//
// ncu on kernel 1b (round 1): the hierarchy walk of a 255-node tree is a chain of 8 levels; levels 0-4 (31 rows) keep ONE
// warp busy while seven wait at the CTA barrier, and that chain (~6 k cycles) is longer than the tile's parallel work.  Here
// two extra warps -- the scouts, alternating tiles -- run up to two tiles AHEAD of the 256 workers (three stages): a scout owns
// the TMA traffic of its tiles (load of tile k, store of tile k-3 out of the same stage: one thread, so the bulk-group waits are
// its own), decides the tile's mark_dirty_trees state, and walks the tile's
// top levels (planner: Tile::top_levels = the leading levels that fit the first 32 rows) in place in the staged tile while
// the workers are still culling the previous tile.  The workers then start at level K: three level rounds instead of eight
// for a binary tree, no dirty-phase barrier, no load/store issue on their path.
//   full[s]  TMA -> everybody        the tile's columns have landed in stage s
//   top[s]   scout -> workers        dirty state + levels < K of stage s are final
//   done[s]  workers -> scout        stage s may be stored and reused
// ------------------------------------------------------------------------------------------
constexpr uint32_t kFull = 0xFFFFFFFFu;
constexpr int kScouts = 2;                       // scout warps per CTA: scout x prepares the CTA's tiles with (index % 2) == x
constexpr int kScoutStages = 3;                  // tile k being culled, tiles k+1 and k+2 being prepared
constexpr int kScoutThreads = kTileRows + 32 * kScouts;
struct __align__(128) ScoutStage {               // the columns that must sit in shared memory: the GlobalTransform tile (walked in place,
    float4 gt0[kWin], gt1[kWin], gt2[kWin];      // stored back in bulk) and the per-row words every phase looks at; Transform and bounds
    uint32_t topo[kWin];                         // are read once per row and come straight from HBM into registers
    uint8_t flags[kWin], state[kWin];
};
struct ScoutSmem {
    ScoutStage st[kScoutStages];
    unsigned long long full[kScoutStages], top[kScoutStages], done[kScoutStages];
    uint16_t parent[kScouts][kTileRows];         // scouts only: the ancestor climb of the slow dirty path
    uint8_t pst[kScoutStages][kTileRows];        // bit0 visited, bit1 gt changed
    uint8_t dirty[kScoutStages][kTileRows];      // TransformTreeChanged, valid when slow[s]
    uint32_t slow[kScoutStages];                 // a row with an in-tile parent changed: workers read dirty[] instead of their own Changed bit
    uint32_t any_gt[kScoutStages];               // a worker row's GlobalTransform changed  \ either one: the tile must be stored
    uint32_t any_top[kScoutStages];              // a row the scout walked changed          /
};
__device__ __forceinline__ void issue_scout_loads(const Rows &R, const Tile &t, ScoutStage &S, unsigned long long *bar) {
    const uint32_t a = t.base & ~15u;
    const uint32_t cnt = ((t.base - a) + t.n_rows + 15u) & ~15u;
    mbar_expect_tx(bar, cnt * (48u + 4u + 2u));
    bulk_g2s(S.gt0, R.gt0 + a, cnt * 16u, bar); bulk_g2s(S.gt1, R.gt1 + a, cnt * 16u, bar); bulk_g2s(S.gt2, R.gt2 + a, cnt * 16u, bar);
    bulk_g2s(S.topo, R.topo + a, cnt * 4u, bar); bulk_g2s(S.flags, R.flags + a, cnt, bar); bulk_g2s(S.state, R.state + a, cnt, bar);
}
__device__ __forceinline__ void issue_scout_store(const Rows &R, const Tile &t, ScoutStage &P) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic smem writes -> async proxy
    const uint32_t poff = t.base & 15u, bytes = (uint32_t)t.n_rows * 16u;
    bulk_s2g(R.gt0 + t.base, P.gt0 + poff, bytes); bulk_s2g(R.gt1 + t.base, P.gt1 + poff, bytes); bulk_s2g(R.gt2 + t.base, P.gt2 + poff, bytes);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void workers_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ bool workers_or(bool p) {
    uint32_t r;
    asm volatile("{\n.reg .pred p, q;\nsetp.ne.u32 p, %1, 0;\nbar.red.or.pred q, 1, 256, p;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(r) : "r"((uint32_t)p) : "memory");
    return r != 0;
}

template <bool CULL, bool SIMPLE, int MINB>
__global__ void __launch_bounds__(kScoutThreads, MINB)
k_propagate_cull_scout(Rows R, const Tile *__restrict__ tiles, uint32_t n_tiles, const __grid_constant__ CullViews cvw,
                       VisibleBufs vb, DevStats *__restrict__ stats, uint32_t static_opt, uint32_t parity) {
    extern __shared__ __align__(128) uint8_t smem_scout[];
    ScoutSmem &s = *reinterpret_cast<ScoutSmem *>(smem_scout);
    const uint32_t tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < kScoutStages; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.top[i], 1); mbar_init(&s.done[i], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");   // PDL: everything above overlapped the previous kernel's tail
    uint32_t n_gt_total = 0, n_vv_total = 0;
    const uint32_t n_mine = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1u) / gridDim.x : 0u;   // tiles of this CTA
    if (tid >= (uint32_t)kTileRows) {
        // ================================ scout warps ================================
        // Scout x prepares tiles x, x+2, x+4, ... of this CTA, two tiles ahead of the workers: per tile it has two of the
        // workers' tile periods for its ~1.3 k instructions (one scout and a one-tile lead made the workers wait, ncu round 2).
        const uint32_t lane = tid & 31u, x = (tid - kTileRows) >> 5;
        for (uint32_t it = x; it < n_mine; it += kScouts) {
            const uint32_t t = blockIdx.x + it * gridDim.x;
            const uint32_t sidx = it % kScoutStages, ph = (it / kScoutStages) & 1u;
            const Tile tile = tiles[t];
            // ---- the stage: tile it-3 lived here; store it once the workers are done with it, then load this tile
            if (it >= (uint32_t)kScoutStages) {
                const uint32_t jt = it - kScoutStages;
                mbar_wait(&s.done[sidx], (jt / kScoutStages) & 1u);
                if (lane == 0 && (s.any_gt[sidx] | s.any_top[sidx])) issue_scout_store(R, tiles[blockIdx.x + jt * gridDim.x], s.st[sidx]);
            }
            if (lane == 0) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");     // this thread's stores have left their stages
                issue_scout_loads(R, tile, s.st[sidx], &s.full[sidx]);
            }
            // the Transform of this lane's row (rows 0..31 hold the tile's top levels): straight from HBM, in flight with the bulk loads
            const uint32_t K = tile.top_levels;
            const bool act = lane < tile.n_rows;
            const uint32_t row = tile.base + lane;
            float4 tA = make_float4(0, 0, 0, 0), tq = tA; float2 tC = make_float2(0, 0);
            if (K > 0 && act) { tA = R.trsA[row]; tq = R.trsB[row]; tC = R.trsC[row]; }
            mbar_wait(&s.full[sidx], ph);
            ScoutStage &S = s.st[sidx];
            const uint32_t off = tile.base & 15u;
            // ---- mark_dirty_trees for the whole tile (systems.rs:111-306): each lane looks at 8 rows
            bool slow = false;
            if (static_opt && R.dirty == nullptr && tile.n_levels > 1) {
                bool mine = false;
#pragma unroll
                for (uint32_t j = 0; j < 8; ++j) {
                    const uint32_t r = lane * 8u + j;
                    if (r < tile.n_rows) mine |= (S.flags[off + r] & F_TCHANGED) && (((S.topo[off + r] >> 9) & 0x1FFu) > 0u);
                }
                slow = __any_sync(kFull, mine);
                if (slow) {       // a row below a root changed: climb the staged parent links
                    for (uint32_t j = 0; j < 8; ++j) {
                        const uint32_t r = lane * 8u + j;
                        if (r < tile.n_rows) {
                            const uint32_t tp = S.topo[off + r];
                            s.parent[x][r] = (uint16_t)((((tp >> 9) & 0x1FFu) > 0u) ? (tp & 0x1FFu) : 0xFFFFu);
                            s.dirty[sidx][r] = 0;
                        }
                    }
                    __syncwarp();
                    for (uint32_t j = 0; j < 8; ++j) {
                        const uint32_t r = lane * 8u + j;
                        if (r < tile.n_rows && (S.flags[off + r] & F_TCHANGED)) {
                            uint32_t c = r;
                            while (!s.dirty[sidx][c]) {       // benign race: every writer stores 1, every chain finishes
                                s.dirty[sidx][c] = 1;
                                const uint32_t p = s.parent[x][c];
                                if (p == 0xFFFFu) break;
                                c = p;
                            }
                        }
                    }
                    __syncwarp();
                }
            }
            if (lane == 0) s.slow[sidx] = slow ? 1u : 0u;
            // ---- the tile's top levels (depth < K), lane = row
            bool top_changed = false;
            if (K > 0) {
                const uint32_t li = off + lane;
                const uint32_t topo = act ? S.topo[li] : T_DETACHED, f = act ? S.flags[li] : 0u;
                const uint32_t depth = (topo >> 9) & 0x1FFu, plocal = topo & 0x1FFu;
                const bool tchanged = f & F_TCHANGED, has_children = topo & T_HAS_CHILDREN;
                const bool in_top = act && !(topo & T_DETACHED) && depth < K;
                bool dirty = tchanged;
                if (static_opt) {
                    if (R.dirty != nullptr) dirty = act && R.dirty[row];
                    else if (slow) dirty = act && s.dirty[sidx][lane];
                }
                const Aff l = affine_from_trs(tA, tq, tC);
                if (act && (topo & T_DETACHED)) s.pst[sidx][lane] = 0;     // never visited, and neither is its subtree
                bool changed = false;
                for (uint32_t lvl = 0; lvl < K; ++lvl) {
                    __syncwarp();
                    if (in_top && depth == lvl) {
                        bool visited = false;
                        Aff n = l;
                        if (depth == 0u) {
                            if (topo & T_ROOT) {
                                visited = has_children ? (!static_opt || dirty) : tchanged;
                                changed = visited;
                            } else {
                                const uint32_t pr = R.parent[row];
                                const uint32_t ps = R.state[pr];
                                visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                                if (visited) {
                                    n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                                    changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);
                                }
                            }
                        } else {
                            const uint32_t pst = s.pst[sidx][plocal];
                            const uint32_t pi = off + plocal;
                            visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                            if (visited) {
                                n.r0 = affine_mul_row(S.gt0[pi], l); n.r1 = affine_mul_row(S.gt1[pi], l); n.r2 = affine_mul_row(S.gt2[pi], l);
                                changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);   // set_if_neq
                            }
                        }
                        if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                        s.pst[sidx][lane] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
                    }
                }
                top_changed = __any_sync(kFull, changed);
            }
            if (lane == 0) s.any_top[sidx] = top_changed ? 1u : 0u;
            __syncwarp();
            if (lane == 0) mbar_arrive(&s.top[sidx]);         // the workers may start this tile
        }
        // ---- the CTA's last three tiles are still in their stages: each scout stores the ones with its parity
        for (uint32_t jt = (n_mine > (uint32_t)kScoutStages ? n_mine - kScoutStages : 0u); jt < n_mine; ++jt) {
            if ((jt % kScouts) != x) continue;
            const uint32_t sj = jt % kScoutStages;
            mbar_wait(&s.done[sj], (jt / kScoutStages) & 1u);
            if (lane == 0 && (s.any_gt[sj] | s.any_top[sj])) issue_scout_store(R, tiles[blockIdx.x + jt * gridDim.x], s.st[sj]);
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    } else {
        // ================================ 256 workers ================================
        const uint32_t lr = tid;
        uint32_t it = 0;
        Tile next_tile = {};
        if (blockIdx.x < n_tiles) next_tile = tiles[blockIdx.x];
        for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
            const uint32_t sidx = it % kScoutStages, ph = (it / kScoutStages) & 1u;
            const Tile tile = next_tile;
            if (t + gridDim.x < n_tiles) next_tile = tiles[t + gridDim.x];    // the next descriptor: in flight during this tile
            const uint32_t off = tile.base & 15u;
            const uint32_t li = off + lr;                 // index into the staged window
            const bool active = lr < tile.n_rows;
            const uint32_t row = tile.base + lr;
            // this row's Transform: read once, so it skips shared memory; requested before the waits below
            float4 tA = make_float4(0, 0, 0, 0), tq = tA; float2 tC = make_float2(0, 0);
            if (active) { tA = R.trsA[row]; tq = R.trsB[row]; tC = R.trsC[row]; }
            mbar_wait(&s.full[sidx], ph);
            mbar_wait(&s.top[sidx], ph);
            ScoutStage &S = s.st[sidx];
            const uint32_t f = active ? S.flags[li] : 0u;
            const uint32_t st8 = active ? S.state[li] : 0u;
            float4 bA = make_float4(0, 0, 0, 0); float2 bB = make_float2(0, 0);
            if (CULL && active) { bA = R.bndA[row]; bB = R.bndB[row]; }
            const uint32_t K = tile.top_levels;
            const uint32_t topo = active ? S.topo[li] : T_DETACHED;
            const uint32_t depth = (topo >> 9) & 0x1FFu, plocal = topo & 0x1FFu;
            const bool tchanged = f & F_TCHANGED;
            const bool has_children = topo & T_HAS_CHILDREN;
            bool dirty = tchanged;
            if (static_opt) {
                if (R.dirty != nullptr) dirty = active && R.dirty[row];
                else if (s.slow[sidx]) dirty = active && s.dirty[sidx][lr];
            }
            const uint32_t my_level = (active && !(topo & T_DETACHED)) ? depth : 0xFFFFFFFFu;
            bool visited = false, changed = false;
            if (my_level < K) {                           // walked by the scout: take its verdict
                const uint32_t pst = s.pst[sidx][lr];
                visited = pst & 1u; changed = pst & 2u;
            } else {
                if (active && (topo & T_DETACHED) && has_children) s.pst[sidx][lr] = 0;
                if (my_level != 0xFFFFFFFFu) {
                    const Aff l = affine_from_trs(tA, tq, tC);
                    if (my_level == 0u) {                 // only when K == 0: roots, flat entities, rows with a parent in another tile
                        Aff n = l;
                        if (topo & T_ROOT) {
                            visited = has_children ? (!static_opt || dirty) : tchanged;
                            changed = visited;
                        } else {
                            const uint32_t pr = R.parent[row];
                            const uint32_t ps = R.state[pr];
                            visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                            if (visited) {
                                n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                                changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);
                            }
                        }
                        if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                        if (has_children) s.pst[sidx][lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
                    }
                    // the loop below needs `l` for the deeper levels: recomputed there (it is cheap) to keep it out of the registers
                }
            }
            {
                const uint32_t first = K > 1u ? K : 1u;
                for (uint32_t lvl = first; lvl < tile.n_levels; ++lvl) {
                    if (!(K > 0u && lvl == K)) {          // the scout's levels are ordered by top[]: no round needed before level K
                        if (lvl < 32u && ((tile.warp_sync_mask >> lvl) & 1u)) __syncwarp(); else workers_sync();
                    }
                    if (my_level == lvl) {
                        const Aff l = affine_from_trs(tA, tq, tC);
                        const uint32_t pst = s.pst[sidx][plocal];
                        const uint32_t pi = off + plocal;
                        visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                        if (visited) {
                            Aff n;   // the parent's rows are the tile's own (in-place) GlobalTransform entries
                            n.r0 = affine_mul_row(S.gt0[pi], l); n.r1 = affine_mul_row(S.gt1[pi], l); n.r2 = affine_mul_row(S.gt2[pi], l);
                            changed = row_neq(n.r0, S.gt0[li]) | row_neq(n.r1, S.gt1[li]) | row_neq(n.r2, S.gt2[li]);   // set_if_neq
                            if (changed) { S.gt0[li] = n.r0; S.gt1[li] = n.r1; S.gt2[li] = n.r2; }
                        }
                        if (has_children) s.pst[sidx][lr] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
                    }
                }
            }
            if (active && tchanged) R.flags[row] = (uint8_t)(f & ~F_TCHANGED);
            uint32_t out = (st8 & (S_VV | S_HAS_CLASS)) | (changed ? S_GT_CHANGED : 0u) | (visited ? S_VISITED : 0u);
            bool vv_changed = false;
            if (CULL) {
                Aff g; g.r0 = S.gt0[li]; g.r1 = S.gt1[li]; g.r2 = S.gt2[li];   // own row: written by this thread, the scout, or untouched
                const bool in_query = active && !(f & F_NO_CPU_CULL);
                const bool base = in_query && (f & F_INHERITED);
        const bool rej_base = base;
                const uint32_t prev = st8 & 1u;
                const uint32_t lane = lr & 31u;
                const bool has_aabb = f & F_AABB;
                const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
                float cx, cy, cz, radius;
                const float hx = bA.w, hy = bB.x, hz = bB.y;
                if (has_aabb) {
                    cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
                    cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
                    cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
                    const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
                    const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
                    const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
                    radius = sqrtf((vx * vx + vy * vy) + vz * vz);
                } else {
                    const bool from_gt = f & F_SPHERE_GT;
                    cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
                    radius = bA.w;
                }
                unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
                if (!SIMPLE && active) {
                    if (R.layers != nullptr) elayers = R.layers[row];
                    if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
                    if (R.rank != nullptr) rnk = R.rank[row];
                }
                // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
                const uint32_t rejmask = warp_view_reject(cvw, rej_base && do_test, rej_base && !do_test, cx, cy, cz, radius);
                bool any = false;
                uint32_t my_ballot = 0;
#pragma unroll
                for (uint32_t v = 0; v < kMaxViews; ++v) {
                    if (v >= cvw.n_views) break;
                    const uint32_t von = cvw.on[v];
                    if (!(von & 1u)) continue;
                    if (SIMPLE && !(von & 4u)) continue;   // bit2: the view includes the default layer
                    if (((rejmask >> v) & 1u) && !(von & 2u)) continue;         // every row of this warp is outside this view's frustum
                    bool vis = base;
                    if (!SIMPLE) {
                        vis = vis && layers_intersect(R, cvw, row, v, elayers);
                        if ((f & F_RANGE) && R.range != nullptr) {
                            const int32_t ri = cvw.range_index[v];
                            vis = vis && ri >= 0 && ((erange >> ri) & 1u);
                        }
                    }
                    if (do_test && !(von & 2u)) {
                        const float d0 = plane_dot_point(cvw.planes[v][0], cx, cy, cz), d1 = plane_dot_point(cvw.planes[v][1], cx, cy, cz);
                        const float d2 = plane_dot_point(cvw.planes[v][2], cx, cy, cz), d3 = plane_dot_point(cvw.planes[v][3], cx, cy, cz);
                        const float d4 = plane_dot_point(cvw.planes[v][4], cx, cy, cz);
                        const bool out_s = (d0 + radius <= 0.0f) | (d1 + radius <= 0.0f) | (d2 + radius <= 0.0f) |
                                           (d3 + radius <= 0.0f) | (d4 + radius <= 0.0f);
                        vis = vis && !out_s;
                        if (vis && has_aabb) {
                            const float d[5] = {d0, d1, d2, d3, d4};
                            bool out_o = false;
#pragma unroll
                            for (int k = 0; k < 5; ++k) {
                                const float4 n = cvw.planes[v][k];
                                const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                                const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                                const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                                const float rr = (dx * hx + dy * hy) + dz * hz;
                                out_o |= (d[k] + rr <= 0.0f);
                            }
                            vis = !out_o;
                        }
                    }
                    any |= vis;
                    const bool listed = vis && (st8 & S_HAS_CLASS);
                    if (SIMPLE || R.rank == nullptr) {
                        const uint32_t b = __ballot_sync(0xFFFFFFFFu, listed);
                        if (lane == v) my_ballot = b;
                    } else if (listed) {
                        uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
                        uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
                        atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                        atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
                    }
                }
                if (my_ballot) {
                    uint32_t *mask = vb.mask + (size_t)lane * vb.words_stride;
                    uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride;
                    const uint32_t row0 = row - lane, w0 = row0 >> 5, sh = row0 & 31u;
                    const uint32_t lo = my_ballot << sh, hi = sh ? (my_ballot >> (32u - sh)) : 0u;
                    if (lo) { atomicOr(mask + w0, lo); atomicAdd(cc + (w0 / kChunkWords), __popc(lo)); }
                    if (hi) { atomicOr(mask + w0 + 1, hi); atomicAdd(cc + ((w0 + 1) / kChunkWords), __popc(hi)); }
                }
                if (in_query) {
                    out = (out & ~S_VV) | (any ? (1u | (prev << 1)) : 0u);
                    vv_changed = (any ? 1u : 0u) != prev;
                    if (vv_changed) out |= S_VV_CHANGED;
                }
                if (R.light_snap != nullptr && (f & F_SPHERE_GT) && active) {
                    const uint32_t ord = R.light_ord[row];     // 0xFFFFFFFF: a sphere-from-GT row that is not a current light
                    if (ord < R.n_lights) R.light_snap[ord] = make_float4(g.r0.w, g.r1.w, g.r2.w, (out & 1u) ? 1.0f : 0.0f);
                }
            } else {
                out |= st8 & S_VV_CHANGED;
            }
            if (active && out != st8) R.state[row] = (uint8_t)out;
            n_gt_total += changed ? 1u : 0u;
            n_vv_total += vv_changed ? 1u : 0u;
            // end of tile: everybody is done with this stage; the scout stores it and reuses the stage
            const bool any_gt = workers_or(changed && !(my_level < K));
            if (lr == 0) { s.any_gt[sidx] = any_gt ? 1u : 0u; mbar_arrive(&s.done[sidx]); }
        }
    }
    // block-reduce the per-thread tallies (warp shuffle, then one shared-memory atomic per warp)
    __shared__ uint32_t s_cnt[2];
    if (tid < 2) s_cnt[tid] = 0;
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { n_gt_total += __shfl_xor_sync(kFull, n_gt_total, o); n_vv_total += __shfl_xor_sync(kFull, n_vv_total, o); }
    if ((tid & 31u) == 0) { if (n_gt_total) atomicAdd(&s_cnt[0], n_gt_total); if (n_vv_total) atomicAdd(&s_cnt[1], n_vv_total); }
    __syncthreads();
    if (tid == 0) {
        if (s_cnt[0]) atomicAdd(&stats->changed[parity][0], s_cnt[0]);
        if (s_cnt[1]) atomicAdd(&stats->changed[parity][1], s_cnt[1]);
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 1w (B200VIS_TILE_KERNEL=warp): the fused propagate -> cull pass with one WARP per tile and no CTA barrier at all.
//
// Why: the CTA-per-tile kernels above spend their time waiting -- the hierarchy walk of a 255-node tree is a chain of
// 8 levels with one warp on the critical path and seven parked at a barrier (ncu round 1: barrier 28 % of stalls, issue
// slots 62 % busy, ~1060 warp instructions per 32 rows of which ~100 only spin through empty level iterations).  Here a
// warp owns a whole tile (<= 256 rows, <= 128 rows with children) and walks it in chunks of 32 schedule slots
// (planner: rows in (depth, row) order, padded so that wide levels start on a chunk boundary).  Per chunk: coalesced
// loads of the 32 rows' columns straight into registers, local affine, one matrix product per level present in the
// chunk (one for all but the top chunk of a tree; __syncwarp between levels), set_if_neq, coalesced store of the changed
// GlobalTransforms, then the cull of the same 32 rows from registers, one ballot per view.  Only rows WITH children
// park their (new) GlobalTransform in shared memory (128 slots of 48 B per warp), where their children find it.
// 32 independent warps per SM hide each other's load latency; nothing ever waits for another warp.
// ------------------------------------------------------------------------------------------
struct __align__(16) WarpSmem {
    float4 g0[kWarpParentSlots], g1[kWarpParentSlots], g2[kWarpParentSlots];
    uint8_t pst[kWarpParentSlots];      // bit0 visited, bit1 gt changed
    uint8_t dirty[kWarpParentSlots];    // TransformTreeChanged of the rows with children (slow path of the dirty phase)
    uint8_t ppar[kWarpParentSlots];     // parent slot of each slot's row, 0xFF = none
};
// byte c (0..7) of the register pair (w0, w1)
__device__ __forceinline__ uint32_t sel_byte(uint32_t w0, uint32_t w1, uint32_t c) { return ((c < 4u ? w0 : w1) >> (8u * (c & 3u))) & 0xFFu; }

// PIPE: the next chunk's columns are loaded into registers while the current chunk is culled (needs ~100 registers);
// !PIPE: they are only prefetched into L2 (no registers), and loaded at the top of their own iteration
template <bool CULL, bool SIMPLE, int MINB, bool PIPE>
__global__ void __launch_bounds__(kTileRows, MINB)
k_tile_warp(Rows R, const WarpTile *__restrict__ tiles, const uint8_t *__restrict__ sched, uint32_t n_tiles,
            const __grid_constant__ CullViews cvw, VisibleBufs vb, DevStats *__restrict__ stats, uint32_t static_opt, uint32_t parity,
            uint32_t *__restrict__ tile_counter) {
    extern __shared__ __align__(16) uint8_t smem_warp[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    WarpSmem &s = reinterpret_cast<WarpSmem *>(smem_warp)[warp];
    asm volatile("griddepcontrol.wait;" ::: "memory");   // PDL: everything above overlapped the previous kernel's tail
    uint32_t n_gt_total = 0, n_vv_total = 0;
    const uint32_t wstride = gridDim.x * (kTileRows / 32);
    uint32_t t = warp * gridDim.x + blockIdx.x;           // consecutive tiles go to different SMs
    if (tile_counter != nullptr) { if (lane == 0) t = atomicAdd(tile_counter, 1u); t = __shfl_sync(kFull, t, 0); }
    while (t < n_tiles) {
        const WarpTile *tp = tiles + t;
        const uint32_t base = tp->base, n_chunks = tp->n_chunks, contig_bits = tp->contig;
        const uint32_t pad = (tp->n_rows == kTileRows) ? 0x100u : 0xFFu;   // a full tile has no padding: 0xFF is local row 255
        const uint8_t *sch = sched + (size_t)tp->sched * kTileRows;
        // ---- the whole schedule and the flag bytes of the tile's rows up front: 8 + 8 independent byte loads per lane, kept
        // packed in four registers (the address chain schedule -> row -> columns is paid once per tile, not per chunk)
        uint32_t sch_w[2] = {0xFFFFFFFFu, 0xFFFFFFFFu}, fl_w[2] = {0u, 0u};
#pragma unroll
        for (uint32_t c = 0; c < (uint32_t)kWarpChunks; ++c)
            if (c < n_chunks) sch_w[c >> 2] = (sch_w[c >> 2] & ~(0xFFu << (8u * (c & 3u)))) | ((uint32_t)sch[c * 32u + lane] << (8u * (c & 3u)));
#pragma unroll
        for (uint32_t c = 0; c < (uint32_t)kWarpChunks; ++c) {
            const uint32_t local = sel_byte(sch_w[0], sch_w[1], c);
            if (c < n_chunks && local != pad) fl_w[c >> 2] |= (uint32_t)R.flags[base + local] << (8u * (c & 3u));
        }
        // ---- mark_dirty_trees (systems.rs:111-306) inside the tile.  Fast path: no row WITH an in-tile parent changed,
        // so every row's TransformTreeChanged bit equals its own Changed<Transform> bit.
        bool slow = false;
        if (static_opt && R.dirty == nullptr) {
            const uint32_t nonroot_l = (lane < (uint32_t)kWarpChunks) ? tp->nonroot[lane] : 0u;
            uint32_t any = 0;
#pragma unroll
            for (uint32_t c = 0; c < (uint32_t)kWarpChunks; ++c) {
                const uint32_t fl = sel_byte(fl_w[0], fl_w[1], c);
                any |= __ballot_sync(kFull, fl & F_TCHANGED) & __shfl_sync(kFull, nonroot_l, c);
            }
            slow = any != 0u;
            if (slow) {
                for (uint32_t c = 0; c < n_chunks; ++c) {       // parent-slot links of the rows with children
                    const uint32_t local = sel_byte(sch_w[0], sch_w[1], c);
                    if (local != pad) {
                        const uint32_t wt = R.wtopo[base + local];
                        if (wt & W_HAS_SLOT) {
                            const uint32_t own = (wt >> 8) & 127u;
                            s.ppar[own] = (uint8_t)((wt & 0xFFu) ? ((wt >> 15) & 127u) : 0xFFu);
                            s.dirty[own] = 0;
                        }
                    }
                }
                __syncwarp();
                for (uint32_t c = 0; c < n_chunks; ++c) {       // every Changed row marks its ancestors
                    const uint32_t local = sel_byte(sch_w[0], sch_w[1], c);
                    const uint32_t fl = sel_byte(fl_w[0], fl_w[1], c);
                    if (local != pad && (fl & F_TCHANGED)) {
                        const uint32_t wt = R.wtopo[base + local];
                        uint32_t sl = (wt & W_HAS_SLOT) ? ((wt >> 8) & 127u) : ((wt & 0xFFu) ? ((wt >> 15) & 127u) : 0xFFu);
                        while (sl != 0xFFu && !s.dirty[sl]) {   // benign race: every writer stores 1, every chain finishes
                            s.dirty[sl] = 1;
                            sl = s.ppar[sl];
                        }
                    }
                }
                __syncwarp();
            }
        }
        // ---- software pipeline over the chunks: the columns of chunk c+1 are requested right after the walk of chunk c and
        // arrive while chunk c is culled (all warps of an SM run the same phases at the same time, so other warps alone do
        // not hide the latency)
        uint32_t n_st = 0, n_wt = T_DETACHED;
        float4 nA = make_float4(0, 0, 0, 0), nq = nA, ng0 = nA, ng1 = nA, ng2 = nA;
        float2 nC = make_float2(0, 0);
        if (PIPE) {
            const uint32_t local = sch_w[0] & 0xFFu;
            if (local != pad) {
                const uint32_t row = base + local;
                n_st = R.state[row]; n_wt = R.wtopo[row];
                nA = R.trsA[row]; nq = R.trsB[row]; nC = R.trsC[row];
                ng0 = R.gt0[row]; ng1 = R.gt1[row]; ng2 = R.gt2[row];
            }
        }
        for (uint32_t c = 0; c < n_chunks; ++c) {
            const uint32_t local = sel_byte(sch_w[0], sch_w[1], c);
            const bool active = local != pad;
            const uint32_t row = base + (active ? local : 0u);
            if (!PIPE) {
                n_st = 0; n_wt = T_DETACHED;
                if (active) {
                    n_st = R.state[row]; n_wt = R.wtopo[row];
                    nA = R.trsA[row]; nq = R.trsB[row]; nC = R.trsC[row];
                    ng0 = R.gt0[row]; ng1 = R.gt1[row]; ng2 = R.gt2[row];
                }
            }
            const uint32_t f = sel_byte(fl_w[0], fl_w[1], c), st8 = n_st, wt = n_wt;
            const float4 A = nA, q = nq;
            const float2 C = nC;
            Aff g; g.r0 = ng0; g.r1 = ng1; g.r2 = ng2;       // current GlobalTransform (old value until overwritten)
            float4 bA = make_float4(0, 0, 0, 0);
            float2 bB = make_float2(0, 0);
            if (CULL && active) { bA = R.bndA[row]; bB = R.bndB[row]; }   // needed after the walk: in flight during it

            const uint32_t depth = wt & 0xFFu, own = (wt >> 8) & 127u, pp = (wt >> 15) & 127u;
            const bool tchanged = f & F_TCHANGED;
            const bool has_children = wt & T_HAS_CHILDREN;     // the reference's "has a Children component"
            const bool has_slot = wt & W_HAS_SLOT;             // ... with children in this tile: they read this row's slot
            bool dirty = tchanged;
            if (static_opt) {
                if (R.dirty != nullptr) dirty = active && R.dirty[row];      // multi-pass plan: k_mark_dirty_global ran first
                else if (slow && has_slot) dirty = tchanged || s.dirty[own];
            }
            const Aff l = affine_from_trs(A, q, C);
            const bool walk = active && !(wt & T_DETACHED);
            // a detached row (ChildOf without a usable parent) is never visited, and neither is its subtree
            if (active && (wt & T_DETACHED) && has_slot) s.pst[own] = 0;
            const uint32_t lo = __reduce_min_sync(kFull, walk ? depth : 0xFFFFu), hi = __reduce_max_sync(kFull, walk ? depth : 0u);
            bool visited = false, changed = false;
            for (uint32_t lvl = lo; lvl <= hi; ++lvl) {        // lo == 0xFFFF (no row to walk) > hi: no iteration
                __syncwarp();                                   // the parents' slots (earlier chunk / lower level) are written
                if (walk && depth == lvl) {
                    Aff n = l;
                    if (depth == 0u) {
                        if (wt & T_ROOT) {
                            // flat entity: sync_simple_transforms (systems.rs:42-79); root with children:
                            // unconditional write (systems.rs:525-530)
                            visited = has_children ? (!static_opt || dirty) : tchanged;
                            changed = visited;
                        } else {                                // parent finished by an earlier pass: read it from HBM
                            const uint32_t pr = R.parent[row];
                            const uint32_t ps = R.state[pr];
                            visited = (ps & S_VISITED) && !(static_opt && !dirty && !(ps & S_GT_CHANGED));
                            if (visited) {
                                n.r0 = affine_mul_row(R.gt0[pr], l); n.r1 = affine_mul_row(R.gt1[pr], l); n.r2 = affine_mul_row(R.gt2[pr], l);
                                changed = row_neq(n.r0, g.r0) | row_neq(n.r1, g.r1) | row_neq(n.r2, g.r2);
                            }
                        }
                    } else {                                    // propagate_descendants_unchecked (systems.rs:706-727)
                        const uint32_t pst = s.pst[pp];
                        visited = (pst & 1u) && !(static_opt && !dirty && !(pst & 2u));
                        if (visited) {
                            n.r0 = affine_mul_row(s.g0[pp], l); n.r1 = affine_mul_row(s.g1[pp], l); n.r2 = affine_mul_row(s.g2[pp], l);
                            changed = row_neq(n.r0, g.r0) | row_neq(n.r1, g.r1) | row_neq(n.r2, g.r2);   // set_if_neq
                        }
                    }
                    if (changed) g = n;
                    if (has_slot) {
                        s.g0[own] = g.r0; s.g1[own] = g.r1; s.g2[own] = g.r2;
                        s.pst[own] = (uint8_t)((visited ? 1u : 0u) | (changed ? 2u : 0u));
                    }
                }
            }
            if (active) {
                if (changed) { R.gt0[row] = g.r0; R.gt1[row] = g.r1; R.gt2[row] = g.r2; }
                if (tchanged) R.flags[row] = (uint8_t)(f & ~F_TCHANGED);
            }
            // request the next chunk's columns: they land while this chunk is culled
            if (PIPE) { n_st = 0; n_wt = T_DETACHED; }
            if (c + 1u < n_chunks) {
                const uint32_t nl = sel_byte(sch_w[0], sch_w[1], c + 1u);
                if (nl != pad) {
                    const uint32_t nrow = base + nl;
                    if (PIPE) {
                        n_st = R.state[nrow]; n_wt = R.wtopo[nrow];
                        nA = R.trsA[nrow]; nq = R.trsB[nrow]; nC = R.trsC[nrow];
                        ng0 = R.gt0[nrow]; ng1 = R.gt1[nrow]; ng2 = R.gt2[nrow];
                    } else if (!(nl & 1u)) {      // one prefetch covers a 32-byte sector: two rows of a float4 column
                        prefetch_l2(R.trsA + nrow); prefetch_l2(R.trsB + nrow); prefetch_l2(R.gt0 + nrow);
                        prefetch_l2(R.gt1 + nrow); prefetch_l2(R.gt2 + nrow);
                        if (CULL) prefetch_l2(R.bndA + nrow);
                    }
                }
            }
            uint32_t out = (st8 & (S_VV | S_HAS_CLASS)) | (changed ? S_GT_CHANGED : 0u) | (visited ? S_VISITED : 0u);
            bool vv_changed = false;
            if (CULL) {
                const bool in_query = active && !(f & F_NO_CPU_CULL);          // Without<NoCpuCulling>
                const bool base_vis = in_query && (f & F_INHERITED);
                const bool rej_base = base_vis;
                const uint32_t prev = st8 & 1u;                                // reset_view_visibility: v = (v&1)<<1
                const bool has_aabb = f & F_AABB;
                const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
                float cx, cy, cz, radius;
                const float hx = bA.w, hy = bB.x, hz = bB.y;
                if (has_aabb) {
                    cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
                    cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
                    cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
                    const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
                    const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
                    const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
                    radius = sqrtf((vx * vx + vy * vy) + vz * vz);
                } else {
                    const bool from_gt = f & F_SPHERE_GT;
                    cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
                    radius = bA.w;
                }
                unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
                if (!SIMPLE && active) {
                    if (R.layers != nullptr) elayers = R.layers[row];
                    if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
                    if (R.rank != nullptr) rnk = R.rank[row];
                }
                // ballot bits map to mask bits when the occupied lanes hold consecutive rows (and rank == row)
                const bool ballots = (SIMPLE || R.rank == nullptr) && ((contig_bits >> c) & 1u);
                // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
                const uint32_t rejmask = warp_view_reject(cvw, rej_base && do_test, rej_base && !do_test, cx, cy, cz, radius);
                bool any = false;
                uint32_t my_ballot = 0;
#pragma unroll
                for (uint32_t v = 0; v < kMaxViews; ++v) {
                    if (v >= cvw.n_views) break;
                    const uint32_t von = cvw.on[v];
                    if (!(von & 1u)) continue;                                 // !camera.is_active (grid-uniform)
                    if (SIMPLE && !(von & 4u)) continue;                       // bit2: the view includes the default layer
                    if (((rejmask >> v) & 1u) && !(von & 2u)) continue;         // every row of this warp is outside this view's frustum
                    bool vis = base_vis;
                    if (!SIMPLE) {
                        vis = vis && layers_intersect(R, cvw, row, v, elayers);
                        if ((f & F_RANGE) && R.range != nullptr) {
                            const int32_t ri = cvw.range_index[v];
                            vis = vis && ri >= 0 && ((erange >> ri) & 1u);
                        }
                    }
                    if (do_test && !(von & 2u)) {
                        // Frustum::intersects_sphere, planes 0..4 (primitives.rs:255-268), branch-free
                        const float d0 = plane_dot_point(cvw.planes[v][0], cx, cy, cz), d1 = plane_dot_point(cvw.planes[v][1], cx, cy, cz);
                        const float d2 = plane_dot_point(cvw.planes[v][2], cx, cy, cz), d3 = plane_dot_point(cvw.planes[v][3], cx, cy, cz);
                        const float d4 = plane_dot_point(cvw.planes[v][4], cx, cy, cz);
                        const bool out_s = (d0 + radius <= 0.0f) | (d1 + radius <= 0.0f) | (d2 + radius <= 0.0f) |
                                           (d3 + radius <= 0.0f) | (d4 + radius <= 0.0f);
                        vis = vis && !out_s;
                        if (vis && has_aabb) {
                            // Frustum::intersects_obb(aabb, affine, true, false) (primitives.rs:272-294)
                            const float d[5] = {d0, d1, d2, d3, d4};
                            bool out_o = false;
#pragma unroll
                            for (int k = 0; k < 5; ++k) {
                                const float4 n = cvw.planes[v][k];   // Aabb::relative_radius (primitives.rs:109-119)
                                const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                                const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                                const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                                const float rr = (dx * hx + dy * hy) + dz * hz;
                                out_o |= (d[k] + rr <= 0.0f);
                            }
                            vis = !out_o;
                        }
                    }
                    any |= vis;
                    // entities without a VisibilityClass are set_visible() but not listed (mod.rs:846-857)
                    const bool listed = vis && (st8 & S_HAS_CLASS);
                    if (ballots) {
                        const uint32_t b = __ballot_sync(kFull, listed);
                        if (lane == v) my_ballot = b;
                    } else if (listed) {
                        uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
                        uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
                        atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                        atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
                    }
                }
                // warp-ballot compaction: lane v publishes view v's bits; the occupied lanes hold consecutive rows, so
                // they touch at most two words of the rank-ordered mask
                const uint32_t occupied = __ballot_sync(kFull, active);
                const uint32_t first = occupied ? (uint32_t)__ffs(occupied) - 1u : 0u;
                const uint32_t row_first = __shfl_sync(kFull, row, first);
                if (my_ballot) {
                    uint32_t *mask = vb.mask + (size_t)lane * vb.words_stride;
                    uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride;
                    const uint32_t bits = my_ballot >> first, w0 = row_first >> 5, sh = row_first & 31u;
                    const uint32_t lo_w = bits << sh, hi_w = sh ? (bits >> (32u - sh)) : 0u;
                    if (lo_w) { atomicOr(mask + w0, lo_w); atomicAdd(cc + (w0 / kChunkWords), __popc(lo_w)); }
                    if (hi_w) { atomicOr(mask + w0 + 1, hi_w); atomicAdd(cc + ((w0 + 1) / kChunkWords), __popc(hi_w)); }
                }
                if (in_query) {
                    // set_visible + mark_newly_hidden_entities_invisible (mod.rs:292-306, 908-918)
                    out = (out & ~S_VV) | (any ? (1u | (prev << 1)) : 0u);
                    vv_changed = (any ? 1u : 0u) != prev;
                    if (vv_changed) out |= S_VV_CHANGED;
                }
                if (R.light_snap != nullptr && (f & F_SPHERE_GT) && active) {
                    const uint32_t ord = R.light_ord[row];     // 0xFFFFFFFF: a sphere-from-GT row that is not a current light
                    if (ord < R.n_lights) R.light_snap[ord] = make_float4(g.r0.w, g.r1.w, g.r2.w, (out & 1u) ? 1.0f : 0.0f);
                }
            } else {
                out |= st8 & S_VV_CHANGED;
            }
            if (active && out != st8) R.state[row] = (uint8_t)out;
            n_gt_total += changed ? 1u : 0u;
            n_vv_total += vv_changed ? 1u : 0u;
        }
        if (tile_counter != nullptr) { if (lane == 0) t = atomicAdd(tile_counter, 1u); t = __shfl_sync(kFull, t, 0); }
        else t += wstride;
    }
    // block-reduce the per-thread tallies (warp shuffle, then one shared-memory atomic per warp)
    __shared__ uint32_t s_cnt[2];
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { n_gt_total += __shfl_xor_sync(kFull, n_gt_total, o); n_vv_total += __shfl_xor_sync(kFull, n_vv_total, o); }
    if (lane == 0) { if (n_gt_total) atomicAdd(&s_cnt[0], n_gt_total); if (n_vv_total) atomicAdd(&s_cnt[1], n_vv_total); }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_cnt[0]) atomicAdd(&stats->changed[parity][0], s_cnt[0]);
        if (s_cnt[1]) atomicAdd(&stats->changed[parity][1], s_cnt[1]);
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 1c: check_visibility as a pure streaming kernel (no hierarchy, no shared memory, no barriers).
// One thread per row, CTAs of 256 rows starting at multiples of 256, so a warp covers exactly one
// 32-bit word of the rank-ordered visible mask: when rows are in Entity::to_bits() order (SIMPLE) the
// ballot is STORED (no atomics, no zeroing of the mask between frames).
// ------------------------------------------------------------------------------------------
template <bool SIMPLE>
__global__ void __launch_bounds__(256, 4)
k_cull(Rows R, const __grid_constant__ CullViews cvw, VisibleBufs vb, DevStats *__restrict__ stats, uint32_t parity) {
    const uint32_t row = blockIdx.x * 256u + threadIdx.x;
    const bool active = row < R.n;
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t f = 0, st8 = 0;
    Aff g; g.r0 = g.r1 = g.r2 = make_float4(0, 0, 0, 0);
    float4 bA = g.r0; float2 bB = make_float2(0, 0);
    if (active) {
        f = R.flags[row]; st8 = R.state[row];
        g.r0 = R.gt0[row]; g.r1 = R.gt1[row]; g.r2 = R.gt2[row];
        bA = R.bndA[row]; bB = R.bndB[row];
    }
    const bool in_query = active && !(f & F_NO_CPU_CULL);
    const bool base = in_query && (f & F_INHERITED);
        const bool rej_base = base;
    const uint32_t prev = st8 & 1u;
    const bool has_aabb = f & F_AABB;
    const bool do_test = (f & (F_AABB | F_SPHERE)) && !(f & F_NO_FRUSTUM);
    float cx, cy, cz, radius;
    const float hx = bA.w, hy = bB.x, hz = bB.y;
    if (has_aabb) {
        cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
        cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
        cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
        const float vx = (g.r0.x * hx + g.r0.y * hy) + g.r0.z * hz;
        const float vy = (g.r1.x * hx + g.r1.y * hy) + g.r1.z * hz;
        const float vz = (g.r2.x * hx + g.r2.y * hy) + g.r2.z * hz;
        radius = sqrtf((vx * vx + vy * vy) + vz * vz);
    } else {
        const bool from_gt = f & F_SPHERE_GT;
        cx = from_gt ? g.r0.w : bA.x; cy = from_gt ? g.r1.w : bA.y; cz = from_gt ? g.r2.w : bA.z;
        radius = bA.w;
    }
    unsigned long long elayers = 1ull; uint32_t erange = 0xFFFFFFFFu, rnk = row;
    if (!SIMPLE && active) {
        if (R.layers != nullptr) elayers = R.layers[row];
        if ((f & F_RANGE) && R.range != nullptr) erange = range_mask_of(R, row, has_aabb, cx, cy, cz, g);
        if (R.rank != nullptr) rnk = R.rank[row];
    }
    // warp-level shortcut: views whose frustum the whole warp's rows are outside of (see warp_view_reject)
    const uint32_t rejmask = warp_view_reject(cvw, rej_base && do_test, rej_base && !do_test, cx, cy, cz, radius);
    bool any = false;
    uint32_t my_ballot = 0;
#pragma unroll
    for (uint32_t v = 0; v < kMaxViews; ++v) {
        if (v >= cvw.n_views) break;
        const uint32_t von = cvw.on[v];
        if (!(von & 1u)) continue;
        if (SIMPLE && !(von & 4u)) { continue; }
        if (((rejmask >> v) & 1u) && !(von & 2u)) continue;         // every row of this warp is outside this view's frustum
        bool vis = base;
        if (!SIMPLE) {
            vis = vis && layers_intersect(R, cvw, row, v, elayers);
            if ((f & F_RANGE) && R.range != nullptr) {
                const int32_t ri = cvw.range_index[v];
                vis = vis && ri >= 0 && ((erange >> ri) & 1u);
            }
        }
        if (do_test && !(von & 2u)) {
            const float d0 = plane_dot_point(cvw.planes[v][0], cx, cy, cz), d1 = plane_dot_point(cvw.planes[v][1], cx, cy, cz);
            const float d2 = plane_dot_point(cvw.planes[v][2], cx, cy, cz), d3 = plane_dot_point(cvw.planes[v][3], cx, cy, cz);
            const float d4 = plane_dot_point(cvw.planes[v][4], cx, cy, cz);
            const bool out_s = (d0 + radius <= 0.0f) | (d1 + radius <= 0.0f) | (d2 + radius <= 0.0f) |
                               (d3 + radius <= 0.0f) | (d4 + radius <= 0.0f);
            vis = vis && !out_s;
            if (vis && has_aabb) {
                const float d[5] = {d0, d1, d2, d3, d4};
                bool out_o = false;
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    const float4 n = cvw.planes[v][k];
                    const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                    const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                    const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                    const float rr = (dx * hx + dy * hy) + dz * hz;
                    out_o |= (d[k] + rr <= 0.0f);
                }
                vis = !out_o;
            }
        }
        any |= vis;
        const bool listed = vis && (st8 & S_HAS_CLASS);
        if (SIMPLE || R.rank == nullptr) {
            const uint32_t b = __ballot_sync(0xFFFFFFFFu, listed);
            if (lane == v) my_ballot = b;
        } else if (listed) {
            uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
            uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
            atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
            atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
        }
    }
    if (SIMPLE || R.rank == nullptr) {
        // lane v owns view v's word: the CTA's rows start at a multiple of 256, so (row - lane) >> 5 is the word
        if (lane < cvw.n_views && (cvw.on[lane] & 1u) && (!SIMPLE || (cvw.on[lane] & 4u))) {
            const uint32_t w0 = (row - lane) >> 5;
            if (w0 < vb.n_words) {
                vb.mask[(size_t)lane * vb.words_stride + w0] = my_ballot;
                if (my_ballot) atomicAdd(vb.chunk_count + ((size_t)parity * kMaxViews + lane) * vb.chunks_stride + (w0 / kChunkWords), __popc(my_ballot));
            }
        }
    }
    uint32_t out = st8;
    bool vv_changed = false;
    if (in_query) {
        out = (st8 & ~(S_VV | S_VV_CHANGED)) | (any ? (1u | (prev << 1)) : 0u);
        vv_changed = (any ? 1u : 0u) != prev;
        if (vv_changed) out |= S_VV_CHANGED;
    } else {
        out = st8 & ~S_VV_CHANGED;
    }
    if (active && out != st8) R.state[row] = (uint8_t)out;
    if (R.light_snap != nullptr && (f & F_SPHERE_GT) && active) {
        const uint32_t ord = R.light_ord[row];
        if (ord < R.n_lights) R.light_snap[ord] = make_float4(g.r0.w, g.r1.w, g.r2.w, (out & 1u) ? 1.0f : 0.0f);
    }
    const uint32_t bv = __ballot_sync(0xFFFFFFFFu, vv_changed);
    if (lane == 0 && bv) atomicAdd(&stats->changed[parity][1], __popc(bv));
}

// mark_dirty_trees for plans whose tiles have parents in other tiles: every Changed row climbs its
// ancestor chain through HBM, stopping at the first already-dirty ancestor (the reference's
// fetch_or early exit, systems.rs:208-223).  `dirty` is zeroed by the caller.
__global__ void k_mark_dirty_global(Rows R) {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= R.n || !(R.flags[row] & F_TCHANGED)) return;
    uint32_t c = row;
    while (true) {
        if (R.dirty[c]) break;
        R.dirty[c] = 1;
        const uint32_t p = R.parent[c];
        if (p >= R.n) break;
        c = p;
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 2: visible mask -> sorted row lists (one CTA per 1024-word chunk per view).
// Output order is ascending rank == ascending Entity::to_bits(): the result of the reference's
// serial `sort_unstable` (visibility/mod.rs:870-874) without a sort.  Also zeroes the mask it
// consumed and the counters of the NEXT frame's parity.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kChunkWords)
k_expand_visible(VisibleBufs vb, DiffBufs db, const uint32_t *__restrict__ row_of_rank, const FrameConsts *__restrict__ fc,
                 DevStats *__restrict__ stats, uint32_t parity, uint32_t n_rows) {
    __shared__ uint32_t s_warp[32], s_diff[32];
    __shared__ uint32_t s_base, s_total;
    const uint32_t v = blockIdx.y, chunk = blockIdx.x, t = threadIdx.x;
    uint32_t *cc = vb.chunk_count + ((size_t)parity * kMaxViews + v) * vb.chunks_stride;
    const uint32_t zslot = (parity + 2u) % 3u;   // the slot frame f+2 will accumulate into
    uint32_t *cc_next = vb.chunk_count + ((size_t)zslot * kMaxViews + v) * vb.chunks_stride;
    // every view of the grid re-arms its counters, also the ones beyond this frame's view count: the count may rise
    // again by frame f+2, and nothing else clears the slot
    if (t == 0) cc_next[chunk] = 0;
    if (chunk == 0 && v == 0 && t < 2) stats->changed[zslot][t] = 0;
    if (v >= fc->n_views) {
        if (db.prev != nullptr && t == 0) db.chunk[(size_t)v * vb.chunks_stride + chunk] = 0;
        return;
    }
    if (!(fc->views[v].flags & 1u)) {         // inactive view: VisibleEntities untouched (mod.rs:780-782)
        if (db.prev != nullptr && t == 0) db.chunk[(size_t)v * vb.chunks_stride + chunk] = 0;   // ... so nothing added / removed
        return;
    }

    const uint32_t word = chunk * kChunkWords + t;
    uint32_t *mask = vb.mask + (size_t)v * vb.words_stride;
    uint32_t w = 0;
    if (word < vb.n_words) { w = mask[word]; if (w) mask[word] = 0; }
    const uint32_t c = __popc(w);
    if (db.prev != nullptr) {
        // the lock-step march of update_cpu_culled_entities (bevy_render/src/view/visibility/mod.rs:194-249) as set
        // algebra on the rank-ordered bit sets: added = new & ~old, removed = old & ~new
        uint32_t a = 0, r = 0;
        if (word < vb.n_words) {
            uint32_t *pv = db.prev + (size_t)v * vb.words_stride + word;
            const uint32_t old = *pv;
            a = w & ~old; r = old & ~w;
            if (old != w) *pv = w;
            db.words[(size_t)v * vb.words_stride + word] = a;
            db.words[((size_t)gridDim.y + v) * vb.words_stride + word] = r;
        }
        uint32_t d = __popc(a) | (__popc(r) << 16);   // a chunk holds 32768 rows: both sums fit 16 bits
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xFFFFFFFFu, d, o);
        if ((t & 31u) == 0) s_diff[t >> 5] = d;
    }
    // block exclusive scan of c
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((t & 31u) >= (uint32_t)o) incl += y; }
    if ((t & 31u) == 31u) s_warp[t >> 5] = incl;
    // base = sum of the counts of the preceding chunks (<= a few hundred values)
    uint32_t part = 0, tot = 0;
    if (t < 32) {
        for (uint32_t i = t; i < vb.n_chunks; i += 32) { const uint32_t x = cc[i]; tot += x; if (i < chunk) part += x; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { part += __shfl_xor_sync(0xFFFFFFFFu, part, o); tot += __shfl_xor_sync(0xFFFFFFFFu, tot, o); }
        if (t == 0) { s_base = part; s_total = tot; }
    }
    __syncthreads();
    if (t < 32) {
        if (db.prev != nullptr) {
            uint32_t d = s_diff[t];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xFFFFFFFFu, d, o);
            if (t == 0) db.chunk[(size_t)v * vb.chunks_stride + chunk] = d;
        }
        uint32_t x = s_warp[t];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (t >= (uint32_t)o) x += y; }
        s_warp[t] = x;   // inclusive over warps
    }
    __syncthreads();
    uint32_t pos = s_base + (incl - c) + ((t >> 5) ? s_warp[(t >> 5) - 1] : 0u);
    uint32_t *out = vb.lists + (size_t)v * vb.list_stride;
    uint8_t *out_cls = vb.classes ? vb.classes + (size_t)v * vb.list_stride : nullptr;
    while (w) {
        const uint32_t b = __ffs(w) - 1; w &= w - 1;
        const uint32_t rk = word * 32u + b;
        const uint32_t rw = row_of_rank ? row_of_rank[rk] : rk;
        if (out_cls) out_cls[pos] = vb.cls[rw];       // one push per class of the row (visibility/mod.rs:852-857): the shim splits
        out[pos++] = rw;
    }
    if (chunk == 0 && t == 0) stats->visible_count[v] = s_total;
    (void)n_rows;
}

// ------------------------------------------------------------------------------------------
// Kernel 2b (SURVEY 8(f) N1): ordered emit of the added / removed rows of each view from the bit sets and per-chunk
// counts k_expand_visible left behind.  Same chunking, one packed (added | removed << 16) block scan.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kChunkWords)
k_emit_visible_diff(VisibleBufs vb, DiffBufs db, const uint32_t *__restrict__ row_of_rank, const FrameConsts *__restrict__ fc) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_base[2], s_total[2];
    const uint32_t v = blockIdx.y, chunk = blockIdx.x, t = threadIdx.x;
    if (v >= fc->n_views || !(fc->views[v].flags & 1u)) {
        if (chunk == 0 && t < 2) db.count[v * 2 + t] = 0;
        return;
    }
    const uint32_t word = chunk * kChunkWords + t;
    uint32_t a = 0, r = 0;
    if (word < vb.n_words) {
        a = db.words[(size_t)v * vb.words_stride + word];
        r = db.words[((size_t)gridDim.y + v) * vb.words_stride + word];
    }
    const uint32_t c = __popc(a) | (__popc(r) << 16);
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((t & 31u) >= (uint32_t)o) incl += y; }
    if ((t & 31u) == 31u) s_warp[t >> 5] = incl;
    if (t < 32) {   // bases: the chunk counts before this one (unpacked: totals may exceed 16 bits)
        const uint32_t *cc = db.chunk + (size_t)v * vb.chunks_stride;
        uint32_t pa = 0, pr = 0, ta = 0, tr = 0;
        for (uint32_t i = t; i < vb.n_chunks; i += 32) {
            const uint32_t x = cc[i], xa = x & 0xFFFFu, xr = x >> 16;
            ta += xa; tr += xr;
            if (i < chunk) { pa += xa; pr += xr; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pa += __shfl_xor_sync(0xFFFFFFFFu, pa, o); pr += __shfl_xor_sync(0xFFFFFFFFu, pr, o);
            ta += __shfl_xor_sync(0xFFFFFFFFu, ta, o); tr += __shfl_xor_sync(0xFFFFFFFFu, tr, o);
        }
        if (t == 0) { s_base[0] = pa; s_base[1] = pr; s_total[0] = ta; s_total[1] = tr; }
    }
    __syncthreads();
    if (t < 32) {
        uint32_t x = s_warp[t];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (t >= (uint32_t)o) x += y; }
        s_warp[t] = x;
    }
    __syncthreads();
    const uint32_t excl = (incl - c) + ((t >> 5) ? s_warp[(t >> 5) - 1] : 0u);
    uint32_t pos_a = s_base[0] + (excl & 0xFFFFu), pos_r = s_base[1] + (excl >> 16);
    uint32_t *out_a = db.lists + (size_t)v * vb.list_stride;
    uint32_t *out_r = db.lists + ((size_t)gridDim.y + v) * vb.list_stride;
    while (a) { const uint32_t b = __ffs(a) - 1; a &= a - 1; const uint32_t rk = word * 32u + b; out_a[pos_a++] = row_of_rank ? row_of_rank[rk] : rk; }
    while (r) { const uint32_t b = __ffs(r) - 1; r &= r - 1; const uint32_t rk = word * 32u + b; out_r[pos_r++] = row_of_rank ? row_of_rank[rk] : rk; }
    if (chunk == 0 && t < 2) db.count[v * 2 + t] = s_total[t];
}
// added / removed rows into the result sink: host_rows[2][max_views][host_stride], host_counts[max_views][2]
__global__ void k_publish_visible_diff(DiffBufs db, uint32_t list_stride, uint32_t *__restrict__ host_rows, uint32_t host_stride,
                                       uint32_t *__restrict__ host_counts, uint32_t n_views, uint32_t max_views) {
    const uint32_t v = blockIdx.y, which = blockIdx.z;
    if (v >= n_views) return;
    const uint32_t n = db.count[v * 2 + which], count = min(n, host_stride);
    const uint32_t *src = db.lists + ((size_t)which * max_views + v) * list_stride;
    uint32_t *dst = host_rows + ((size_t)which * max_views + v) * host_stride;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) dst[i] = src[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) host_counts[v * 2 + which] = n;
}

// ------------------------------------------------------------------------------------------
// Kernel 3: assign_objects_to_clusters, point lights: one warp per (light, view)
// (crates/bevy_light/src/cluster/assign.rs:487-748).  Lanes split the (z, y) rows of the
// iterative sphere refinement; each row sets its [min_x, max_x] bits in the cluster x light mask.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 mat4_mul_point(const float *m, float x, float y, float z) {   // M * (p, 1)
    float4 r;   // (((X*x) + (Y*y)) + (Z*z)) + (W*1)
    r.x = ((m[0] * x + m[4] * y) + m[8] * z) + m[12] * 1.0f;
    r.y = ((m[1] * x + m[5] * y) + m[9] * z) + m[13] * 1.0f;
    r.z = ((m[2] * x + m[6] * y) + m[10] * z) + m[14] * 1.0f;
    r.w = ((m[3] * x + m[7] * y) + m[11] * z) + m[15] * 1.0f;
    return r;
}
// view_z_to_z_slice (assign.rs:1046-1062) through the host-computed thresholds on u = -view_z
__device__ __forceinline__ uint32_t z_slice_of(const float *thr, uint32_t z_slices, float view_z) {
    const float u = -view_z;
    uint32_t lo = 0, hi = z_slices - 1;       // number of k in [1, z_slices) with u >= thr[k-1]
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (u >= thr[mid]) lo = mid + 1; else hi = mid; }
    return lo;
}
// ndc_position_to_cluster (assign.rs:922-941)
__device__ __forceinline__ uint3 ndc_to_cluster(const DevClusterView &cv, const float *thr, float nx, float ny, float view_z) {
    const float fx = gl_min(gl_max(nx * 0.5f + 0.5f, 0.0f), 1.0f);
    const float fy = gl_min(gl_max(ny * -0.5f + 0.5f, 0.0f), 1.0f);
    const uint32_t x = __float2uint_rz(floorf(fx * (float)cv.dims[0]));
    const uint32_t y = __float2uint_rz(floorf(fy * (float)cv.dims[1]));
    const uint32_t z = z_slice_of(thr, cv.dims[2], view_z);
    return make_uint3(min(x, cv.dims[0] - 1), min(y, cv.dims[1] - 1), min(z, cv.dims[2] - 1));
}

constexpr uint32_t kStagedPlanes = 512;   // plane tables up to this many entries are staged in shared memory

// One light against one view's froxel grid, executed by a warp (lanes split the (z, y) rows): frustum test, view-space
// AABB -> cluster range, iterative sphere refinement; `set(ci)` is called for every cluster the light touches.  Returns
// false if the light is rejected before the grid walk; `far_out` (lane 0) receives the light's farthest_z candidate.
struct ClusterTables { const float *thr; const float4 *xp, *yp, *zp; };
template <typename SetBit>
__device__ __forceinline__ bool assign_one_light(const DevClusterView &cv, const ClusterTables &tb, float px, float py, float pz, float range,
                                                 uint32_t lane, float &far_out, uint32_t &count, SetBit set) {
#pragma unroll
    for (int k = 0; k < 6; ++k)                                         // frustum.intersects_sphere(.., true)
        if (plane_dot_point(cv.frustum[k], px, py, pz) + range <= 0.0f) return false;
    const float *thr = tb.thr;
    const bool ortho = cv.is_ortho;
    // cluster_space_clusterable_object_aabb (assign.rs:948-1036)
    const float4 vc = mat4_mul_point(cv.vfw, px, py, pz);
    const float hx = range * fabsf(cv.scale[0]), hy = range * fabsf(cv.scale[1]), hz = range * fabsf(cv.scale[2]);
    const float minx = vc.x - hx, miny = vc.y - hy, maxx = vc.x + hx, maxy = vc.y + hy;
    const float minz = fminf(vc.z - hz, -1.17549435e-38f), maxz = fminf(vc.z + hz, -1.17549435e-38f);
    float nminx, nminy, nmaxx, nmaxy;
    {
        const float4 a = mat4_mul_point(cv.cfv, minx, miny, minz), b = mat4_mul_point(cv.cfv, minx, miny, maxz);
        const float4 c = mat4_mul_point(cv.cfv, maxx, maxy, minz), d = mat4_mul_point(cv.cfv, maxx, maxy, maxz);
        const float ax = a.x / a.w, ay = a.y / a.w, bx = b.x / b.w, by = b.y / b.w;
        const float cx = c.x / c.w, cy = c.y / c.w, dx = d.x / d.w, dy = d.y / d.w;
        nminx = gl_min(gl_min(gl_min(ax, bx), cx), dx); nminy = gl_min(gl_min(gl_min(ay, by), cy), dy);
        nmaxx = gl_max(gl_max(gl_max(ax, bx), cx), dx); nmaxy = gl_max(gl_max(gl_max(ay, by), cy), dy);
        nminx = gl_min(gl_max(nminx, -1.0f), 1.0f); nminy = gl_min(gl_max(nminy, -1.0f), 1.0f);
        nmaxx = gl_min(gl_max(nmaxx, -1.0f), 1.0f); nmaxy = gl_min(gl_max(nmaxy, -1.0f), 1.0f);
    }
    const uint3 c0 = ndc_to_cluster(cv, thr, nminx, nminy, minz), c1 = ndc_to_cluster(cv, thr, nmaxx, nmaxy, maxz);
    const uint3 lo = make_uint3(min(c0.x, c1.x), min(c0.y, c1.y), min(c0.z, c1.z));
    const uint3 hi = make_uint3(max(c0.x, c1.x), max(c0.y, c1.y), max(c0.z, c1.z));
    // view-space sphere (assign.rs:551-556)
    const float sr = range * cv.scale_max;
    {
        // farthest_z (assign.rs:558-561): -row2 . (t,1) + range*scale.z ; fmax against 0
        const float4 r2 = make_float4(cv.vfw[2], cv.vfw[6], cv.vfw[10], cv.vfw[14]);
        far_out = -plane_dot_point(r2, px, py, pz) + range * cv.scale[2];
    }
    const float4 cc = mat4_mul_point(cv.cfv, vc.x, vc.y, vc.z);
    const float ndx = cc.x / cc.w, ndy = cc.y / cc.w, ndz = cc.z / cc.w;
    const uint3 ccl = ndc_to_cluster(cv, thr, ndx, ndy, vc.z);
    const bool has_zc = ndz <= 1.0f; const uint32_t zc = ccl.z;
    bool has_yc; uint32_t yc = 0;
    if (ndy > 1.0f) has_yc = false;
    else if (ndy < -1.0f) { has_yc = true; yc = cv.dims[1] + 1; }
    else { has_yc = true; yc = ccl.y; }

    const float4 *xp = tb.xp, *yp = tb.yp, *zp = tb.zp;
    const uint32_t ny = hi.y - lo.y + 1, npairs = (hi.z - lo.z + 1) * ny;
    for (uint32_t p = lane; p < npairs; p += 32) {
        const uint32_t z = lo.z + p / ny, y = lo.y + p % ny;
        float ox = vc.x, oy = vc.y, oz = vc.z, orad = sr;
        if (!has_zc || z != zc) {                                  // project_to_plane_z (assign.rs:1094-1113)
            const float4 pl = (has_zc && z < zc) ? zp[z + 1] : zp[z];
            const float zz = pl.w / pl.z;
            const float dist = zz - oz;
            if (fabsf(dist) > orad) continue;
            oz = zz;
            orad = sqrtf(orad * orad - dist * dist);
        }
        if (!has_yc || y != yc) {                                  // project_to_plane_y (assign.rs:1116-1134)
            const float4 pl = (has_yc && y < yc) ? yp[y + 1] : yp[y];
            const float dist = ortho ? pl.w - oy : -(oy * pl.y + oz * pl.z);
            if (fabsf(dist) > orad) continue;
            ox = ox + dist * pl.x; oy = oy + dist * pl.y; oz = oz + dist * pl.z;
            orad = sqrtf(orad * orad - dist * dist);
        }
        uint32_t min_x = lo.x;                                     // assign.rs:647-675, get_distance_x :1081-1091
        while (true) {
            if (min_x >= hi.x) break;
            const float4 pl = xp[min_x + 1];
            const float dx = ortho ? ox - pl.w : pl.x * ox + pl.z * oz;
            if (-dx + orad > 0.0f) break;
            ++min_x;
        }
        uint32_t max_x = hi.x;
        while (true) {
            if (max_x <= min_x) break;
            const float4 pl = xp[max_x];
            const float dx = ortho ? ox - pl.w : pl.x * ox + pl.z * oz;
            if (dx + orad > 0.0f) break;
            --max_x;
        }
        uint32_t ci = (y * cv.dims[0] + min_x) * cv.dims[2] + z;   // assign.rs:676-678
        for (uint32_t x = min_x; x <= max_x; ++x) { set(ci); ci += cv.dims[2]; }
        count += max_x - min_x + 1;
    }
    return true;
}

__global__ void __launch_bounds__(256)
k_cluster_assign(Rows R, Lights L, const FrameConsts *__restrict__ fc, ClusterBufs cb, DevStats *__restrict__ stats) {
    __shared__ float4 s_planes[kStagedPlanes];
    __shared__ float s_thr[kStagedPlanes];
    const uint32_t v = blockIdx.y;
    if (v >= fc->n_views) return;
    const DevClusterView &cv = fc->cviews[v];
    if (!cv.enabled) return;
    // stage this view's x/y/z plane tables and z thresholds once per CTA (all 8 warps share the view)
    const uint32_t nx = cv.dims[0] + 1, ny_p = cv.dims[1] + 1, nz = cv.dims[2] + 1;
    const bool staged = nx + ny_p + nz <= kStagedPlanes;
    if (staged) {
        const float4 *gx = reinterpret_cast<const float4 *>(cb.blob + cv.x_off);
        const float4 *gy = reinterpret_cast<const float4 *>(cb.blob + cv.y_off);
        const float4 *gz = reinterpret_cast<const float4 *>(cb.blob + cv.z_off);
        for (uint32_t i = threadIdx.x; i < nx; i += 256) s_planes[i] = gx[i];
        for (uint32_t i = threadIdx.x; i < ny_p; i += 256) s_planes[nx + i] = gy[i];
        for (uint32_t i = threadIdx.x; i < nz; i += 256) s_planes[nx + ny_p + i] = gz[i];
        for (uint32_t i = threadIdx.x; i + 1 < cv.dims[2]; i += 256) s_thr[i] = cb.blob[cv.thr_off + i];
        __syncthreads();
    }
    const uint32_t li = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (li >= L.n) return;
    float px, py, pz;
    if (L.snap != nullptr) {                                            // snapshot taken right after the tile pass
        const float4 sp = L.snap[li];
        if (sp.w == 0.0f) return;                                       // view_visibility.get() (assign.rs:195)
        px = sp.x; py = sp.y; pz = sp.z;
    } else {
        const uint32_t row = L.row[li];
        if (!(R.state[row] & 1u)) return;                               // view_visibility.get() (assign.rs:195)
        px = R.gt0[row].w; py = R.gt1[row].w; pz = R.gt2[row].w;        // GlobalTransform::translation
    }
    const unsigned long long ll = L.layers ? L.layers[li] : 1ull;
    if (!(cv.layer_mask & ll)) return;                                  // assign.rs:489
    const float range = L.range[li];
    ClusterTables tb;
    tb.thr = staged ? s_thr : cb.blob + cv.thr_off;
    tb.xp = staged ? s_planes : reinterpret_cast<const float4 *>(cb.blob + cv.x_off);
    tb.yp = staged ? s_planes + nx : reinterpret_cast<const float4 *>(cb.blob + cv.y_off);
    tb.zp = staged ? s_planes + nx + ny_p : reinterpret_cast<const float4 *>(cb.blob + cv.z_off);
    uint32_t *mask = cb.send + ((size_t)v * cb.words + (li >> 5)) * kMaxClusters;
    const uint32_t bit = 1u << (li & 31u);
    uint32_t count = 0;
    float this_far = 0.0f;
    if (!assign_one_light(cv, tb, px, py, pz, range, lane, this_far, count, [&](uint32_t ci) { atomicOr(mask + ci, bit); })) return;
    // farthest_z candidates accumulate in the slab's trailer (values > 0 only: integer max == float max)
    if (lane == 0 && this_far > 0.0f) atomicMax(cb.send + (cb.slab_words - kMaxViews) + v, __float_as_uint(this_far));
    (void)count; (void)stats;
}

// ------------------------------------------------------------------------------------------
// Kernel 3+4 fused (single GPU): assign_objects_to_clusters for one view in ONE launch by a thread-block CLUSTER.
// The view's cluster x light bit matrix lives in the distributed shared memory of the cluster's CTAs: CTA j owns the
// clusters [j * per, (j+1) * per) (all mask words of those clusters), every CTA takes a share of the LIGHTS and sets
// bits with shared-memory atomics in whichever CTA owns the cluster (DSMEM).  After a cluster barrier each CTA
// popcounts its own clusters, the CTA totals are exchanged through DSMEM, and every CTA emits its part of the CSR:
// no global bit matrix, no clear kernel, no re-count.  Ascending light ordinal per cluster = the reference's push order
// (the outer loop runs over lights, assign.rs:487).
// ------------------------------------------------------------------------------------------
constexpr uint32_t kFusedThreads = 1024;
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_nctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t dsmem_addr(const void *p, uint32_t cta) {       // shared::cluster address of p in CTA `cta`
    uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(cta));
    return r;
}
__device__ __forceinline__ void dsmem_or(uint32_t addr, uint32_t v) {
    asm volatile("red.relaxed.cluster.shared::cluster.or.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t dsmem_ld(uint32_t addr) {
    uint32_t v; asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v;
}

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__global__ void __launch_bounds__(kFusedThreads)
k_cluster_fused(Rows R, Lights L, const FrameConsts *__restrict__ fc, ClusterBufs cb, DevStats *__restrict__ stats) {
    extern __shared__ __align__(16) uint8_t smem_fused[];
    __shared__ float4 s_planes[kStagedPlanes];
    __shared__ float s_thr[kStagedPlanes];
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_total, s_far, s_base, s_farmax;
    const uint32_t v = blockIdx.y, t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    const uint32_t rank = cluster_ctarank(), nrank = cluster_nctarank();
    uint32_t *offsets = cb.offsets + (size_t)v * (kMaxClusters + 1);
    // early outs are uniform over the cluster (they depend on the view only): nobody is left waiting at a cluster barrier
    if (v >= fc->n_views) return;
    const DevClusterView &cv = fc->cviews[v];
    if (!cv.enabled) {
        if (rank == 0 && t == 0) { offsets[0] = 0; stats->cl_overflow[v] = 0; stats->cl_index_count[v] = 0; stats->cl_farthest_bits[v] = 0; }
        return;
    }
    if (cb.p2p && L.per_rank) {     // light records pushed by the peers (k_record_push): wait for every rank's stamp of this frame
        if (t < cb.world) {
            const uint32_t *flag = cb.peer_flags[cb.rank] + cb.xparity * cb.world + t;
            uint32_t spins = 0;
            while ((int32_t)(ld_acquire_sys(flag) - cb.stamp) < 0) {
                __nanosleep(64);
                if (++spins > (1u << 22)) { stats->cl_overflow[v] = 2u; break; }   // a peer never arrived (~0.3 s): report, do not hang
            }
        }
        __syncthreads();
    }
    const uint32_t nc = cv.n_clusters, per = (nc + nrank - 1) / nrank, words = (L.n + 31u) / 32u;
    uint32_t *s_mask = reinterpret_cast<uint32_t *>(smem_fused);      // [words][per]
    for (uint32_t i = t; i < words * per; i += kFusedThreads) s_mask[i] = 0;
    if (t == 0) { s_total = 0; s_far = 0; }
    const uint32_t nx = cv.dims[0] + 1, ny_p = cv.dims[1] + 1, nz = cv.dims[2] + 1;
    const bool staged = nx + ny_p + nz <= kStagedPlanes;
    if (staged) {
        const float4 *gx = reinterpret_cast<const float4 *>(cb.blob + cv.x_off);
        const float4 *gy = reinterpret_cast<const float4 *>(cb.blob + cv.y_off);
        const float4 *gz = reinterpret_cast<const float4 *>(cb.blob + cv.z_off);
        for (uint32_t i = t; i < nx; i += kFusedThreads) s_planes[i] = gx[i];
        for (uint32_t i = t; i < ny_p; i += kFusedThreads) s_planes[nx + i] = gy[i];
        for (uint32_t i = t; i < nz; i += kFusedThreads) s_planes[nx + ny_p + i] = gz[i];
        for (uint32_t i = t; i + 1 < cv.dims[2]; i += kFusedThreads) s_thr[i] = cb.blob[cv.thr_off + i];
    }
    cluster_sync_all();                    // every CTA's matrix is zeroed before the first remote bit arrives
    ClusterTables tb;
    tb.thr = staged ? s_thr : cb.blob + cv.thr_off;
    tb.xp = staged ? s_planes : reinterpret_cast<const float4 *>(cb.blob + cv.x_off);
    tb.yp = staged ? s_planes + nx : reinterpret_cast<const float4 *>(cb.blob + cv.y_off);
    tb.zp = staged ? s_planes + nx + ny_p : reinterpret_cast<const float4 *>(cb.blob + cv.z_off);
    // ---- assign: light li is handled by warp (li / nrank) % 32 of CTA li % nrank
    for (uint32_t li = rank + nrank * warp; li < L.n; li += nrank * (kFusedThreads / 32)) {
        float px, py, pz;
        if (L.snap != nullptr || L.per_rank) {
            const float4 sp = light_snap_of(L, li);
            if (sp.w == 0.0f) continue;                                     // view_visibility.get() (assign.rs:195); unused slot
            px = sp.x; py = sp.y; pz = sp.z;
        } else {
            const uint32_t row = L.row[li];
            if (!(R.state[row] & 1u)) continue;
            px = R.gt0[row].w; py = R.gt1[row].w; pz = R.gt2[row].w;
        }
        const unsigned long long ll = light_layers_of(L, li);
        if (!(cv.layer_mask & ll)) continue;                                // assign.rs:489
        const uint32_t bit = 1u << (li & 31u), wbase = (li >> 5) * per;
        uint32_t count = 0;
        float this_far = 0.0f;
        const bool in = assign_one_light(cv, tb, px, py, pz, light_range_of(L, li), lane, this_far, count, [&](uint32_t ci) {
            const uint32_t owner = ci / per;
            dsmem_or(dsmem_addr(&s_mask[wbase + (ci - owner * per)], owner), bit);
        });
        if (in && lane == 0 && this_far > 0.0f) atomicMax(&s_far, __float_as_uint(this_far));
    }
    cluster_sync_all();                    // all bits of all lights have landed
    // ---- popcount -> scan -> ordered emit, per owned cluster
    const uint32_t first = rank * per, c = first + t;
    uint32_t cnt = 0;
    if (t < per && c < nc)
        for (uint32_t w = 0; w < words; ++w) cnt += __popc(s_mask[w * per + t]);
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= (uint32_t)o) incl += y; }
    if (lane == 31u) s_warp[warp] = incl;
    __syncthreads();
    if (t < 32) {
        uint32_t x = s_warp[t];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (t >= (uint32_t)o) x += y; }
        s_warp[t] = x;          // inclusive over warps
        if (t == 31) s_total = x;
    }
    cluster_sync_all();                    // every CTA's total (and farthest-z candidate) is published
    if (t < 32) {
        uint32_t tot_r = 0, far_r = 0;
        if (t < nrank) { tot_r = dsmem_ld(dsmem_addr(&s_total, t)); far_r = dsmem_ld(dsmem_addr(&s_far, t)); }
        uint32_t b = (t < rank) ? tot_r : 0u, fm = far_r;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
            fm = max(fm, __shfl_xor_sync(0xFFFFFFFFu, fm, o));
        }
        if (t == 0) { s_base = b; s_farmax = fm; }
    }
    // this CTA has read its peers' shared memory; the matching wait sits at the very end, so that no CTA exits (and
    // frees its shared memory) while a peer may still be reading it, and the emit below overlaps the barrier
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    __syncthreads();
    const uint32_t base = s_base;
    uint32_t pos = base + (incl - cnt) + (warp ? s_warp[warp - 1] : 0u);
    uint32_t *indices = cb.indices + (size_t)v * cb.index_cap;
    if (t < per && c < nc) {
        offsets[c] = pos;
        for (uint32_t w = 0; w < words; ++w) {
            uint32_t m = s_mask[w * per + t];
            while (m) {
                const uint32_t b = __ffs(m) - 1; m &= m - 1;
                if (pos < cb.index_cap) indices[pos] = w * 32u + b;
                ++pos;
            }
        }
        if (c == nc - 1) {                // the CTA holding the last cluster publishes the totals
            offsets[nc] = pos;
            stats->cl_overflow[v] = pos > cb.index_cap ? 1u : 0u;
            stats->cl_index_count[v] = pos;                  // every (cluster, light) pair is one index: the reference's count
        }
    }
    if (rank == 0 && t == 0) stats->cl_farthest_bits[v] = s_farmax;
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ------------------------------------------------------------------------------------------
// Kernel 4: cluster x light bitmask (all ranks' slabs) -> per-cluster ordered index lists.
// kListBlocks CTAs per view, 1024 clusters each: popcount -> scan -> ordered emit.  A CTA gets the
// offset of its first cluster by re-counting the clusters before it (L2-resident words, coalesced),
// which is cheaper than a second launch or a cross-CTA hand-over.  Ascending (rank, light) order
// is the reference's push order (the outer loop runs over lights, assign.rs:487).
// ------------------------------------------------------------------------------------------
constexpr uint32_t kListBlocks = kMaxClusters / 1024;

// ------------------------------------------------------------------------------------------
// Kernel 3b: the cluster exchange as peer stores.  Instead of an ncclAllGather of the cluster x light slabs, every rank
// WRITES the words of its slab that are in use straight into every rank's gathered buffer over NVLink (buffers of the
// other processes are mapped through CUDA IPC), then publishes a per-(parity, rank) stamp with system-scope release
// semantics; k_cluster_lists spins on the stamps of all ranks (acquire) before it reads.  Two parities: a rank can be
// at most one frame ahead of the slowest one, because its next-but-one push comes after its own list build, which
// waited for everybody's stamp of the frame in between.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_slab_push(const FrameConsts *__restrict__ fc, ClusterBufs cb, uint32_t *__restrict__ done) {
    const uint32_t v = blockIdx.y;
    const size_t slab_words = cb.slab_words;
    if (blockIdx.x == 0 && threadIdx.x < cb.world && v < kMaxViews) {   // the trailer: this view's farthest_z candidate
        const size_t tr = ((size_t)cb.xparity * cb.world + cb.rank) * slab_words + (slab_words - kMaxViews) + v;
        cb.peer[threadIdx.x][tr] = cb.send[(slab_words - kMaxViews) + v];
    }
    if (v < fc->n_views && fc->cviews[v].enabled) {
        const uint32_t nc = fc->cviews[v].n_clusters;
        const uint32_t *mine = cb.send + (size_t)v * cb.words * kMaxClusters;
        const size_t dst0 = ((size_t)cb.xparity * cb.world + cb.rank) * slab_words + (size_t)v * cb.words * kMaxClusters;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cb.words * nc; i += gridDim.x * blockDim.x) {
            const uint32_t w = i / nc, c = i - w * nc;
            const uint32_t val = mine[(size_t)w * kMaxClusters + c];
            for (uint32_t r = 0; r < cb.world; ++r) cb.peer[r][dst0 + (size_t)w * kMaxClusters + c] = val;
        }
    }
    // last CTA out publishes the stamp: every CTA's stores are fenced at system scope before it counts itself in
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t total = gridDim.x * gridDim.y;
        if (atomicAdd(done, 1u) == total - 1u) {
            *done = 0;
            __threadfence_system();
            for (uint32_t r = 0; r < cb.world; ++r) st_release_sys(cb.peer_flags[r] + cb.xparity * cb.world + cb.rank, cb.stamp);
        }
    }
}

// The light-record exchange as peer stores: CTA r copies this rank's light block (28 bytes per light) into rank r's gathered
// buffer and stamps it; k_cluster_fused waits for every rank's stamp of the frame before it reads a light.
__global__ void __launch_bounds__(256)
k_record_push(const uint32_t *__restrict__ block, uint32_t block_words, ClusterBufs cb) {
    const uint32_t r = blockIdx.x;
    uint32_t *dst = cb.peer[r] + ((size_t)cb.xparity * cb.world + cb.rank) * cb.slab_words;
    for (uint32_t i = threadIdx.x; i < block_words; i += blockDim.x) dst[i] = block[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) st_release_sys(cb.peer_flags[r] + cb.xparity * cb.world + cb.rank, cb.stamp);
}

__global__ void __launch_bounds__(1024)
k_cluster_lists(const FrameConsts *__restrict__ fc, ClusterBufs cb, DevStats *__restrict__ stats) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_red[32];
    const uint32_t v = blockIdx.y, blk = blockIdx.x, t = threadIdx.x;
    if (v >= fc->n_views) return;
    const DevClusterView &cv = fc->cviews[v];
    uint32_t *offsets = cb.offsets + (size_t)v * (kMaxClusters + 1);
    const uint32_t nc = cv.enabled ? cv.n_clusters : 0u;
    if (cb.p2p) {   // wait until every rank's slab of this frame has landed in this rank's gathered buffer
        // (spinning here, in the 16 CTAs of the list build, measured faster than a separate one-warp wait kernel: one
        // scheduling delay on a GPU that is busy with the next frame's tile pass instead of two)
        if (t < cb.world) {
            const uint32_t *flag = cb.peer_flags[cb.rank] + cb.xparity * cb.world + t;
            uint32_t spins = 0;
            while ((int32_t)(ld_acquire_sys(flag) - cb.stamp) < 0) {
                __nanosleep(64);
                if (++spins > (1u << 22)) { stats->cl_overflow[v] = 2u; break; }   // a peer never arrived (~0.3 s): report, do not hang
            }
        }
        __syncthreads();
    }
    if (blk == 0 && t == 0 && !cv.enabled) { offsets[0] = 0; stats->cl_overflow[v] = 0; }
    const size_t rank_stride = cb.slab_words;
    const uint32_t *base = cb.recv + (size_t)v * cb.words * kMaxClusters;
    uint32_t *indices = cb.indices + (size_t)v * cb.index_cap;
    const uint32_t first = blk * 1024u;
    // (a) this thread's cluster; (b) its share of the clusters in front of this CTA
    const uint32_t c = first + t;
    uint32_t cnt = 0, before = 0;
    if (c < nc)
        for (uint32_t r = 0; r < cb.world; ++r)
            for (uint32_t w = 0; w < cb.words; ++w) cnt += __popc(base[r * rank_stride + (size_t)w * kMaxClusters + c]);
    for (uint32_t p = t; p < first && p < nc; p += 1024)
        for (uint32_t r = 0; r < cb.world; ++r)
            for (uint32_t w = 0; w < cb.words; ++w) before += __popc(base[r * rank_stride + (size_t)w * kMaxClusters + p]);
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((t & 31u) >= (uint32_t)o) incl += y; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xFFFFFFFFu, before, o);
    if ((t & 31u) == 31u) s_warp[t >> 5] = incl;
    if ((t & 31u) == 0u) s_red[t >> 5] = before;
    __syncthreads();
    if (t < 32) {
        uint32_t x = s_warp[t], b = s_red[t];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (t >= (uint32_t)o) x += y; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
        s_warp[t] = x;          // inclusive over warps
        if (t == 0) s_red[0] = b;
    }
    __syncthreads();
    uint32_t pos = s_red[0] + (incl - cnt) + ((t >> 5) ? s_warp[(t >> 5) - 1] : 0u);
    if (c < nc) {
        offsets[c] = pos;
        for (uint32_t r = 0; r < cb.world; ++r)
            for (uint32_t w = 0; w < cb.words; ++w) {
                uint32_t m = base[r * rank_stride + (size_t)w * kMaxClusters + c];
                while (m) {
                    const uint32_t b = __ffs(m) - 1; m &= m - 1;
                    if (pos < cb.index_cap) indices[pos] = r * cb.max_lights + w * 32u + b;
                    ++pos;
                }
            }
    }
    // the CTA holding the last cluster publishes the total; CTA 0 publishes / re-arms the accumulators
    if (nc && c == nc - 1) {
        offsets[nc] = pos;
        if (!(cb.p2p && stats->cl_overflow[v] == 2u)) stats->cl_overflow[v] = pos > cb.index_cap ? 1u : 0u;
    }
    if (nc && c == nc - 1) stats->cl_index_count[v] = pos;     // every (cluster, light) pair is one index: the reference's count
    if (blk == 0 && t == 0) {
        if (!nc) stats->cl_index_count[v] = 0;
        uint32_t far = 0;                                       // max over the ranks' candidates (gathered trailers)
        for (uint32_t r = 0; r < cb.world; ++r) far = max(far, cb.recv[r * rank_stride + (rank_stride - kMaxViews) + v]);
        stats->cl_farthest_bits[v] = far;
    }
    // NOTE: the slab is zeroed for the next frame by k_cluster_clear (a CTA here may still be re-counting it)
}

// set_lights: write each light's ordinal into the per-row light_ord column (cleared to 0xFFFFFFFF by the caller) so that the
// tile kernel can publish the light snapshot itself; *all_tagged is cleared if some light row is not a sphere-from-GT row or
// two lights share a row (then the separate snapshot kernel is used instead)
__global__ void k_tag_lights(Rows R, Lights L, uint32_t *__restrict__ light_ord, uint32_t *__restrict__ all_tagged) {
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= L.n) return;
    const uint32_t row = L.row[li];
    if (row < R.n && (R.flags[row] & F_SPHERE_GT) && !(R.flags[row] & F_AABB)) {
        if (atomicCAS(light_ord + row, 0xFFFFFFFFu, li) != 0xFFFFFFFFu) *all_tagged = 0;
    } else {
        *all_tagged = 0;
    }
}

// (pos, visible) of every light, copied right after the tile pass so that the cluster kernels of frame f can run
// on a side stream while frame f+1's tile pass already rewrites GlobalTransform / ViewVisibility
__global__ void k_snapshot_lights(Rows R, Lights L, float4 *__restrict__ snap) {
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= L.n) return;
    const uint32_t row = L.row[li];
    snap[li] = make_float4(R.gt0[row].w, R.gt1[row].w, R.gt2[row].w, (R.state[row] & 1u) ? 1.0f : 0.0f);
}

// GlobalTransform::radius_vec3a(h) = (matrix3 * h).length() (global_transform.rs:252-254) on the row form of the matrix:
// Mat3A * Vec3A = ((X*h.x) + (Y*h.y)) + (Z*h.z) lane-wise, Vec3A::length = sqrt((x*x + y*y) + z*z) -- the expression the
// cull phase evaluates for an Aabb's half extents (glam order unverified, DESIGN.md §5)
__device__ __forceinline__ float radius_vec3a(float4 r0, float4 r1, float4 r2, float hx, float hy, float hz) {
    const float vx = (r0.x * hx + r0.y * hy) + r0.z * hz;
    const float vy = (r1.x * hx + r1.y * hy) + r1.z * hz;
    const float vz = (r2.x * hx + r2.y * hy) + r2.z * hz;
    return sqrtf((vx * vx + vy * vy) + vz * vz);
}

// The clusterable objects of b200vis_set_clusterable_objects at the light snapshot's stream position: (translation, visible)
// of ordinal base + j into `snap`, and the radius of the kinds that derive it from GlobalTransform into `range`
// (assign.rs:256-295).  Rect-light ranges were written into every frame slot at set time.
__global__ void k_snapshot_objects(Rows R, ClusterObjects O, float4 *__restrict__ snap, float *__restrict__ range) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= O.n) return;
    const uint32_t row = O.row[j], kind = O.kind[j];
    const float4 r0 = R.gt0[row], r1 = R.gt1[row], r2 = R.gt2[row];
    snap[O.base + j] = make_float4(r0.w, r1.w, r2.w, (R.state[row] & 1u) ? 1.0f : 0.0f);
    if (kind == kKindReflectionProbe || kind == kKindIrradianceVolume) {
        range[O.base + j] = radius_vec3a(r0, r1, r2, 1.0f, 1.0f, 1.0f);           // transform.radius_vec3a(Vec3A::ONE)
    } else if (kind == kKindDecal) {
        // transform.scale().length() (global_transform.rs:240-248): the axis lengths, the first one times copysign(1, det),
        // whose sign squares away exactly -- so the determinant is not needed
        const float lx = sqrtf((r0.x * r0.x + r1.x * r1.x) + r2.x * r2.x);
        const float ly = sqrtf((r0.y * r0.y + r1.y * r1.y) + r2.y * r2.y);
        const float lz = sqrtf((r0.z * r0.z + r1.z * r1.z) + r2.z * r2.z);
        range[O.base + j] = sqrtf((lx * lx + ly * ly) + lz * lz);
    }
}

// ---- result sink: coalesced copies of a frame's results into mapped pinned host memory ----------------------
// visible lists: grid (blocks, views), grid-stride over the view's count
__global__ void k_publish_visible(const uint32_t *__restrict__ lists, uint32_t list_stride, const DevStats *__restrict__ stats,
                                  uint32_t *__restrict__ host_rows, uint32_t host_stride, uint32_t n_views,
                                  const uint8_t *__restrict__ classes, uint8_t *__restrict__ host_classes) {
    const uint32_t v = blockIdx.y;
    if (v >= n_views) return;
    const uint32_t count = min(stats->visible_count[v], host_stride);
    // one row per thread: a warp writes 128 contiguous bytes (view strides need not be 16-byte multiples)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x)
        host_rows[(size_t)v * host_stride + i] = lists[(size_t)v * list_stride + i];
    if (host_classes != nullptr && classes != nullptr)      // 4 class bytes per thread: 128 contiguous bytes per warp
        for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) * 4u; i < count; i += gridDim.x * blockDim.x * 4u)
            for (uint32_t k = i; k < min(i + 4u, count); ++k) host_classes[(size_t)v * host_stride + k] = classes[(size_t)v * list_stride + k];
}
// cluster CSR + the stats block (also formats b200vis_frame_stats, whose layout the host passes as offsets)
__global__ void k_publish_clusters(const FrameConsts *__restrict__ fc, const uint32_t *__restrict__ offsets, const uint32_t *__restrict__ indices,
                                   uint32_t index_cap, uint32_t *__restrict__ host_offsets, uint32_t *__restrict__ host_indices,
                                   uint32_t host_cap, const DevStats *__restrict__ stats, uint32_t *__restrict__ host_stats,
                                   uint32_t changed_slot, uint32_t frame) {
    const uint32_t v = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
    if (v == 0 && blockIdx.x == 0 && host_stats != nullptr) {
        // b200vis_frame_stats: visible_count[8] cluster_index_count[8] cluster_farthest_z[8] overflow[8] gt vv frame pad
        if (threadIdx.x < 8) {
            host_stats[threadIdx.x] = stats->visible_count[threadIdx.x];
            host_stats[8 + threadIdx.x] = stats->cl_index_count[threadIdx.x];
            host_stats[16 + threadIdx.x] = stats->cl_farthest_bits[threadIdx.x];
            host_stats[24 + threadIdx.x] = stats->cl_overflow[threadIdx.x];
        }
        if (threadIdx.x == 8) { host_stats[32] = stats->changed[changed_slot][0]; host_stats[33] = stats->changed[changed_slot][1]; host_stats[34] = frame; host_stats[35] = 0; }
    }
    if (v >= fc->n_views || host_offsets == nullptr) return;
    const DevClusterView &cv = fc->cviews[v];
    const uint32_t nc = cv.enabled ? cv.n_clusters : 0u;
    const uint32_t *off = offsets + (size_t)v * (kMaxClusters + 1);
    if (t <= nc) host_offsets[(size_t)v * (kMaxClusters + 1) + t] = off[t];
    const uint32_t total = min(min(off[nc], index_cap), host_cap);
    for (uint32_t i = t; i < total; i += gridDim.x * blockDim.x) host_indices[(size_t)v * host_cap + i] = indices[(size_t)v * index_cap + i];
}

// ---- column write-back: the frame's GlobalTransform / ViewVisibility results into the caller's ECS columns (mapped host
// memory, PCIe posted writes).  One warp per 128 rows: the state bytes are read four at a time, the change flags travel as
// bit sets, a ViewVisibility word crosses PCIe only when one of its four bytes differs from what the host already holds
// (device-side shadow), and the changed rows' matrices are transposed through shared memory so that every store
// instruction covers up to 512 contiguous bytes of the host column (whole PCIe write bursts).
template <int STRIDE>
__global__ void __launch_bounds__(256)
k_writeback_columns(Rows R, float *__restrict__ host_gt, uint32_t *__restrict__ host_gt_bits, uint8_t *__restrict__ host_vv,
                    uint32_t *__restrict__ host_vv_bits, uint8_t *__restrict__ vv_shadow) {
    __shared__ float4 s_t[8][32 * (STRIDE / 4)];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t n_groups = (R.n + 127u) / 128u, n_words = (R.n + 31u) / 32u;
    for (uint32_t grp = blockIdx.x * 8u + warp; grp < n_groups; grp += gridDim.x * 8u) {
        const uint32_t r4 = grp * 128u + lane * 4u;          // this lane's four rows (the state column is padded past n)
        uint32_t st4 = (r4 < R.n) ? *reinterpret_cast<const uint32_t *>(R.state + r4) : 0u;
        if (r4 + 3u >= R.n) st4 &= (r4 >= R.n) ? 0u : (0xFFFFFFFFu >> (8u * (3u - (R.n - 1u - r4))));   // bytes past the last row
        if (host_vv != nullptr && r4 < R.n) {
            const uint32_t vv4 = st4 & 0x03030303u;
            uint32_t *sh = reinterpret_cast<uint32_t *>(vv_shadow + r4);
            if (*sh != vv4) {
                *sh = vv4;
                if (r4 + 3u < R.n && (reinterpret_cast<uintptr_t>(host_vv) & 3u) == 0u) *reinterpret_cast<uint32_t *>(host_vv + r4) = vv4;
                else for (uint32_t j = 0; j < 4u && r4 + j < R.n; ++j) host_vv[r4 + j] = (uint8_t)(vv4 >> (8u * j));   // tail / unaligned column
            }
        }
        // change bits: bit j of the lane's nibble = row r4 + j; eight lanes make one 32-row word
        uint32_t g = ((st4 >> 4) & 1u) | ((st4 >> 11) & 2u) | ((st4 >> 18) & 4u) | ((st4 >> 25) & 8u);
        uint32_t v = ((st4 >> 5) & 1u) | ((st4 >> 12) & 2u) | ((st4 >> 19) & 4u) | ((st4 >> 26) & 8u);
        g <<= 4u * (lane & 7u); v <<= 4u * (lane & 7u);
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { g |= __shfl_xor_sync(0xFFFFFFFFu, g, o); v |= __shfl_xor_sync(0xFFFFFFFFu, v, o); }
        const uint32_t w = grp * 4u + (lane >> 3);
        if ((lane & 7u) == 0u && w < n_words) {
            if (host_gt_bits != nullptr) host_gt_bits[w] = g;
            if (host_vv_bits != nullptr) host_vv_bits[w] = v;
        }
        if (host_gt == nullptr) continue;
        constexpr int Q = STRIDE / 4;                         // float4 per row in the host layout
#pragma unroll 1
        for (uint32_t j = 0; j < 4; ++j) {
            const uint32_t gbits = __shfl_sync(0xFFFFFFFFu, g, j * 8u);
            if (!gbits) continue;
            const uint32_t row = grp * 128u + j * 32u + lane;
            if ((gbits >> lane) & 1u) {
                const float4 a = R.gt0[row], b = R.gt1[row], c = R.gt2[row];
                float4 *o = &s_t[warp][lane * Q];
                if (STRIDE == 16) {                           // glam Affine3A: x_axis, y_axis, z_axis, translation as Vec3A
                    o[0] = make_float4(a.x, b.x, c.x, 0.0f); o[1] = make_float4(a.y, b.y, c.y, 0.0f);
                    o[2] = make_float4(a.z, b.z, c.z, 0.0f); o[3] = make_float4(a.w, b.w, c.w, 0.0f);
                } else {                                      // packed X.xyz Y.xyz Z.xyz T.xyz
                    o[0] = make_float4(a.x, b.x, c.x, a.y); o[1] = make_float4(b.y, c.y, a.z, b.z);
                    o[2] = make_float4(c.z, a.w, b.w, c.w);
                }
            }
            __syncwarp();
            float4 *dst = reinterpret_cast<float4 *>(host_gt) + ((size_t)grp * 128u + j * 32u) * Q;
#pragma unroll
            for (int k = 0; k < Q; ++k) {
                const uint32_t idx = k * 32u + lane;          // consecutive lanes -> consecutive 16-byte pieces of the column
                if ((gbits >> (idx / Q)) & 1u) dst[idx] = s_t[warp][idx];
            }
            __syncwarp();
        }
    }
}

// zero this rank's slab for the next frame's assign kernel (only the words in use)
__global__ void k_cluster_clear(const FrameConsts *__restrict__ fc, ClusterBufs cb) {
    const uint32_t v = blockIdx.y;
    if (v >= fc->n_views) return;
    const DevClusterView &cv = fc->cviews[v];
    if (!cv.enabled) return;
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0) cb.send[(cb.slab_words - kMaxViews) + v] = 0;
    if (c >= cv.n_clusters) return;
    uint32_t *mine = cb.send + (size_t)v * cb.words * kMaxClusters;
    for (uint32_t w = 0; w < cb.words; ++w) mine[(size_t)w * kMaxClusters + c] = 0;
}

// ------------------------------------------------------------------------------------------
// Kernels 5a-c (SURVEY 8(f) N3): check_point_light_mesh_visibility for point lights
// (crates/bevy_light/src/lib.rs:517-668).  One thread per row loops over the frame's shadow lights (staged through
// shared memory a few at a time): layers / visibility-range gates, Sphere::intersects_obb against the light's range
// sphere (primitives.rs:219-226), then Frustum::intersects_obb with near and far planes on each of the six cubemap
// faces (primitives.rs:272-294).  Visible (row, light, face) triples go into rank-ordered bit sets that
// k_expand_shadow turns into the sorted CubemapVisibleEntities lists; a row seen by any light gets
// ViewVisibility::set_visible (visibility/mod.rs:292-306) applied on top of what the camera cull left.
// ------------------------------------------------------------------------------------------
constexpr int kShadowChunk = 4;   // items staged per round (4 x 608 B)
// a point / spot light takes part only if it is in some view's VisibleEntities (lib.rs:561-563): its rank bit in the per-view
// sets; directional cascades are pre-filtered by the caller (shadow_maps_enabled && visible, lib.rs:395-399)
__global__ void k_shadow_select(ShadowBufs sb, const uint32_t *__restrict__ rank, const uint32_t *__restrict__ view_sets,
                                uint32_t words_stride, uint32_t n_views) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= sb.n_lights) return;
    if (sb.lights[s].kind == 2u) { sb.active[s] = 1; return; }
    const uint32_t row = sb.lights[s].row, rk = rank ? rank[row] : row;
    uint32_t on = 0;
    for (uint32_t v = 0; v < n_views; ++v) on |= (view_sets[(size_t)v * words_stride + (rk >> 5)] >> (rk & 31u)) & 1u;
    sb.active[s] = on;
}
__global__ void __launch_bounds__(256)
k_shadow_cull(Rows R, ShadowBufs sb, uint32_t words_stride, uint32_t chunks_stride, DevStats *__restrict__ stats,
              uint32_t changed_slot) {
    __shared__ ShadowLight s_light[kShadowChunk];
    __shared__ float4 s_sphere[kShadowChunk];
    __shared__ uint32_t s_on[kShadowChunk];
    const uint32_t row = blockIdx.x * 256u + threadIdx.x, lane = threadIdx.x & 31u;
    const bool active = row < R.n;
    uint32_t f = 0, st8 = 0, erange = 0;
    Aff g; g.r0 = g.r1 = g.r2 = make_float4(0, 0, 0, 0);
    float4 bA = g.r0; float2 bB = make_float2(0, 0);
    bool eligible = false;
    unsigned long long elayers = 1ull;
    uint32_t rnk = row;
    if (active) {
        f = R.flags[row]; st8 = R.state[row];
        eligible = sb.caster[row] && !(f & F_NO_CPU_CULL) && (f & F_INHERITED);
        if (eligible) {
            g.r0 = R.gt0[row]; g.r1 = R.gt1[row]; g.r2 = R.gt2[row];
            bA = R.bndA[row]; bB = R.bndB[row];
            if (R.layers != nullptr) elayers = R.layers[row];
            if ((f & F_RANGE) && sb.has_ranges && R.range != nullptr) erange = R.range[row];
        }
        if (R.rank != nullptr) rnk = R.rank[row];
    }
    const bool ranged = (f & F_RANGE) && sb.has_ranges;   // gated on one bit of the VisibleEntityRanges mask (lib.rs:607-616, 432-441)
    const bool has_aabb = f & F_AABB, no_fc = f & F_NO_FRUSTUM;
    const float hx = bA.w, hy = bB.x, hz = bB.y;
    // transform_point3a(aabb.center)
    const float cx = ((g.r0.x * bA.x + g.r0.y * bA.y) + g.r0.z * bA.z) + g.r0.w;
    const float cy = ((g.r1.x * bA.x + g.r1.y * bA.y) + g.r1.z * bA.z) + g.r1.w;
    const float cz = ((g.r2.x * bA.x + g.r2.y * bA.y) + g.r2.z * bA.z) + g.r2.w;
    // ---- block pre-pass: an axis-aligned box around the world-space centres of this CTA's bounded candidate rows and the largest
    // OBB reach E1 = sum_i h_i * |axis_i|_1 among them (>= relative_radius(v) / |v| for every direction v).  An item whose range
    // sphere (or, for a cascade, one of whose half spaces) cannot reach the box is skipped for the whole CTA: every exact per-row
    // test would fail.  Rows are spatially coherent (a CTA holds one tree), so almost every (CTA, light) pair goes this way.
    __shared__ float s_red[8][7];
    __shared__ float s_box[7];
    const float e1_row = fabsf(hx) * ((fabsf(g.r0.x) + fabsf(g.r1.x)) + fabsf(g.r2.x)) + fabsf(hy) * ((fabsf(g.r0.y) + fabsf(g.r1.y)) + fabsf(g.r2.y)) +
                         fabsf(hz) * ((fabsf(g.r0.z) + fabsf(g.r1.z)) + fabsf(g.r2.z));
    // rows without an Aabb / with NoFrustumCulling pass without a test, rows with non-finite numbers behave arbitrarily in the
    // exact tests: either kind switches the skipping off for its CTA
    const bool bounded = eligible && has_aabb && !no_fc && isfinite(((cx + cy) + cz) + e1_row);
    const int unbounded_any = __syncthreads_or(eligible && !bounded);
    {
        const float inf = __int_as_float(0x7f800000);
        float v[7];
        v[0] = bounded ? cx : inf; v[1] = bounded ? cy : inf; v[2] = bounded ? cz : inf;
        v[3] = bounded ? -cx : inf; v[4] = bounded ? -cy : inf; v[5] = bounded ? -cz : inf;       // min of the negation = -max
        v[6] = bounded ? -e1_row : inf;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[k] = fminf(v[k], __shfl_xor_sync(0xFFFFFFFFu, v[k], o));
            if (lane == 0) s_red[threadIdx.x >> 5][k] = v[k];
        }
        __syncthreads();
        if (threadIdx.x < 7) {
            float m = s_red[0][threadIdx.x];
            for (int w = 1; w < 8; ++w) m = fminf(m, s_red[w][threadIdx.x]);
            s_box[threadIdx.x] = m;
        }
    }
    // ---- which items can reach this CTA at all: one thread per item tests the block box (nothing else does per-item work)
    constexpr uint32_t kLiveWords = 8;                               // up to 256 items are pre-tested; further items are always live
    __shared__ uint32_t s_live[kLiveWords];
    if (threadIdx.x < kLiveWords) s_live[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < sb.n_lights; i += 256u) {
        bool live = sb.active[i] != 0u;
        if (live && !unbounded_any && i < 32u * kLiveWords) {
            const ShadowLight &sl = sb.lights[i];
            const float bx0 = s_box[0], by0 = s_box[1], bz0 = s_box[2], bx1 = -s_box[3], by1 = -s_box[4], bz1 = -s_box[5], e1 = -s_box[6];
            bool skip = !(bx0 <= bx1);                               // no bounded candidate row in this CTA at all
            if (!skip && sl.kind < 2u) {
                // light_sphere = (GlobalTransform translation, range) (lib.rs:575-578, 680-683)
                const float sx = R.gt0[sl.row].w, sy = R.gt1[sl.row].w, sz = R.gt2[sl.row].w;
                const float dx = fmaxf(fmaxf(bx0 - sx, sx - bx1), 0.0f), dy = fmaxf(fmaxf(by0 - sy, sy - by1), 0.0f);
                const float dz = fmaxf(fmaxf(bz0 - sz, sz - bz1), 0.0f);
                const float reach = (sl.range + e1) * 1.001f + 1e-3f;      // d <= r + rr/d <= r + E1 where the exact test passes
                skip = (dx * dx + dy * dy) + dz * dz > reach * reach;
            } else if (!skip) {
                for (int k = 0; k < 6 && !skip; ++k) {               // a half space no point of the box reaches, even grown by E1
                    if (k == 4) continue;
                    const float4 n = sl.planes[0][k];
                    const float m = ((fmaxf(n.x * bx0, n.x * bx1) + fmaxf(n.y * by0, n.y * by1)) + fmaxf(n.z * bz0, n.z * bz1)) + n.w;
                    skip = m + (e1 * 1.001f + 1e-3f) * ((fabsf(n.x) + fabsf(n.y)) + fabsf(n.z)) < 0.0f;
                }
            }
            live = !skip;
        }
        if (live && i < 32u * kLiveWords) atomicOr(&s_live[i >> 5], 1u << (i & 31u));
    }
    __syncthreads();
    bool any = false;
    for (uint32_t i0 = 0; i0 < sb.n_lights; ++i0) {
        if (i0 < 32u * kLiveWords) {                                 // jump to the next live item (CTA-uniform)
            uint32_t w = s_live[i0 >> 5] >> (i0 & 31u);
            if (!w) { i0 |= 31u; continue; }
            i0 += (uint32_t)__ffs(w) - 1u;
        } else if (!sb.active[i0]) continue;
        __syncthreads();
        for (uint32_t q = threadIdx.x; q < sizeof(ShadowLight) / 16; q += 256u)
            reinterpret_cast<float4 *>(s_light)[q] = reinterpret_cast<const float4 *>(sb.lights + i0)[q];
        if (threadIdx.x == 0) {
            const ShadowLight &sl = sb.lights[i0];
            s_sphere[0] = sl.kind < 2u ? make_float4(R.gt0[sl.row].w, R.gt1[sl.row].w, R.gt2[sl.row].w, sl.range) : make_float4(0, 0, 0, 0);
        }
        __syncthreads();
        {
            const uint32_t i = 0, s0 = i0;
            const ShadowLight &sl = s_light[i];
            const uint32_t kind = sl.kind, n_faces = kind == 0u ? 6u : 1u;
            bool in = eligible && (sl.layers & elayers) != 0ull;
            if (in && ranged) in = sl.range_index >= 0 && sl.range_index < 32 && ((erange >> sl.range_index) & 1u);
            uint32_t faces = kind == 0u ? 0x3Fu : 1u;                // no Aabb: pushed to every list of the item (lib.rs:639-645)
            if (in && has_aabb && !no_fc) {
                if (kind < 2u) {
                    // Sphere::intersects_obb: d_sq <= radius * d + relative_radius(v) (primitives.rs:219-226)
                    const float4 sp = s_sphere[i];
                    const float vx = cx - sp.x, vy = cy - sp.y, vz = cz - sp.z;
                    const float d_sq = (vx * vx + vy * vy) + vz * vz, d = sqrtf(d_sq);
                    const float ax = fabsf(dot3(vx, vy, vz, g.r0.x, g.r1.x, g.r2.x));
                    const float ay = fabsf(dot3(vx, vy, vz, g.r0.y, g.r1.y, g.r2.y));
                    const float az = fabsf(dot3(vx, vy, vz, g.r0.z, g.r1.z, g.r2.z));
                    const float rr = (ax * hx + ay * hy) + az * hz;
                    in = d_sq <= sp.w * d + rr;
                }
                if (in) {
                    faces = 0;
                    for (uint32_t fc = 0; fc < n_faces; ++fc) {
                        bool inside = true;
#pragma unroll
                        for (int k = 0; k < 6; ++k) {   // cubemap faces and spot lights test near and far; cascades skip the near plane (lib.rs:455-458)
                            if (k == 4 && kind == 2u) continue;
                            const float4 n = sl.planes[fc][k];
                            const float dx = fabsf(dot3(n.x, n.y, n.z, g.r0.x, g.r1.x, g.r2.x));
                            const float dy = fabsf(dot3(n.x, n.y, n.z, g.r0.y, g.r1.y, g.r2.y));
                            const float dz = fabsf(dot3(n.x, n.y, n.z, g.r0.z, g.r1.z, g.r2.z));
                            const float prr = (dx * hx + dy * hy) + dz * hz;
                            inside = inside && !(plane_dot_point(n, cx, cy, cz) + prr <= 0.0f);
                        }
                        faces |= inside ? (1u << fc) : 0u;
                    }
                }
            }
            if (!in) faces = 0;
            any |= faces != 0u;
            if (__any_sync(0xFFFFFFFFu, faces != 0u)) {
                for (uint32_t fc = 0; fc < n_faces; ++fc) {
                    const uint32_t list = (s0 + i) * 6u + fc;
                    uint32_t *mask = sb.mask + (size_t)list * words_stride;
                    uint32_t *cc = sb.chunk_count + (size_t)list * chunks_stride;
                    if (R.rank == nullptr) {
                        const uint32_t b = __ballot_sync(0xFFFFFFFFu, (faces >> fc) & 1u);
                        if (lane == 0 && b) { mask[row >> 5] = b; atomicAdd(cc + ((row >> 5) / kChunkWords), __popc(b)); }
                    } else if ((faces >> fc) & 1u) {
                        atomicOr(mask + (rnk >> 5), 1u << (rnk & 31u));
                        atomicAdd(cc + ((rnk >> 5) / kChunkWords), 1u);
                    }
                }
            }
        }
    }
    // set_visible on top of the camera cull's result.  A row the cameras left hidden has state 0 (+ S_VV_CHANGED when it was
    // visible last frame): visible now means (1 | prev << 1), and the change flag fires iff it was NOT visible last frame.
    if (any && !(st8 & 1u)) {
        const uint32_t prev = (st8 & S_VV_CHANGED) ? 1u : 0u;
        const uint32_t out = (st8 & ~(S_VV | S_VV_CHANGED)) | 1u | (prev << 1) | (prev ? 0u : S_VV_CHANGED);
        R.state[row] = (uint8_t)out;
        atomicAdd(&stats->changed[changed_slot][1], prev ? 0xFFFFFFFFu : 1u);
    }
}
// the sorted CubemapVisibleEntities lists from the bit sets (same chunked scan as k_expand_visible)
__global__ void __launch_bounds__(kChunkWords)
k_expand_shadow(ShadowBufs sb, uint32_t n_words, uint32_t n_chunks, uint32_t words_stride, uint32_t chunks_stride,
                const uint32_t *__restrict__ row_of_rank) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_base, s_total;
    const uint32_t item = blockIdx.y, chunk = blockIdx.x, t = threadIdx.x;
    const uint32_t n_faces = sb.lights[item].kind == 0u ? 6u : 1u;
    for (uint32_t face = 0; face < 6u; ++face) {
        const uint32_t list = item * 6u + face;
        if (face >= n_faces) { if (chunk == 0 && t == 0) sb.count[list] = 0; continue; }
        const uint32_t *cc = sb.chunk_count + (size_t)list * chunks_stride;
        // almost every (list, chunk) is empty (a light reaches a few trees): its mask words are all zero, nothing to read or emit
        if (chunk != 0 && cc[chunk] == 0) continue;
        const uint32_t word = chunk * kChunkWords + t;
        uint32_t *mask = sb.mask + (size_t)list * words_stride;
        uint32_t w = 0;
        if (word < n_words) { w = mask[word]; if (w) mask[word] = 0; }
        const uint32_t c = __popc(w);
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((t & 31u) >= (uint32_t)o) incl += y; }
        __syncthreads();                       // the previous face's readers of s_warp / s_base are done
        if ((t & 31u) == 31u) s_warp[t >> 5] = incl;
        if (t < 32) {
            uint32_t part = 0, tot = 0;
            for (uint32_t i = t; i < n_chunks; i += 32) { const uint32_t x = cc[i]; tot += x; if (i < chunk) part += x; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { part += __shfl_xor_sync(0xFFFFFFFFu, part, o); tot += __shfl_xor_sync(0xFFFFFFFFu, tot, o); }
            if (t == 0) { s_base = part; s_total = tot; }
        }
        __syncthreads();
        if (t < 32) {
            uint32_t x = s_warp[t];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (t >= (uint32_t)o) x += y; }
            s_warp[t] = x;
        }
        __syncthreads();
        uint32_t pos = s_base + (incl - c) + ((t >> 5) ? s_warp[(t >> 5) - 1] : 0u);
        uint32_t *out = sb.lists + (size_t)list * sb.list_cap;
        while (w) {
            const uint32_t b = __ffs(w) - 1; w &= w - 1;
            const uint32_t rk = word * 32u + b;
            if (pos < sb.list_cap) out[pos] = row_of_rank ? row_of_rank[rk] : rk;
            ++pos;
        }
        if (chunk == 0 && t == 0) sb.count[list] = s_total;
    }
}

// ------------------------------------------------------------------------------------------
// Kernel 4b (SURVEY 8(f) N2): Clusters -> ViewClusterBindings.  The reference walks a record stream
// (ClusterHeader, Light, Light, ..., bevy_pbr/src/cluster/mod.rs:419-470) and pushes offsets-and-counts / indices
// one by one (:494-520, :609-697); with the CSR already on the device every output word is independent.
// ------------------------------------------------------------------------------------------
__global__ void k_pack_cluster_bindings(const FrameConsts *__restrict__ fc, ClusterBufs cb, BindingBufs bb) {
    constexpr uint32_t kMaxIndices = 16384u;               // ViewClusterBindings::MAX_INDICES (:587)
    constexpr uint32_t kUniformWords = 16384u / 4u;        // MAX_UNIFORM_ITEMS uvec4 = 4096 u32 (:585-586)
    constexpr uint32_t kCountSize = 9u;                    // CLUSTER_COUNT_SIZE (:43)
    const uint32_t v = blockIdx.y;
    if (v >= fc->n_views) return;
    const DevClusterView &cv = fc->cviews[v];
    const uint32_t nc = cv.enabled ? cv.n_clusters : 0u;
    const uint32_t *off = cb.offsets + (size_t)v * (kMaxClusters + 1);
    const uint32_t *idx = cb.indices + (size_t)v * cb.index_cap;
    const uint32_t total = nc ? off[nc] : 0u, avail = min(total, cb.index_cap);
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    uint32_t *oc = bb.oc + (size_t)v * kMaxClusters * 8, *il = bb.il + (size_t)v * bb.il_stride;
    auto gpu_index = [&](uint32_t ordinal) -> uint32_t {
        if (bb.map == nullptr) return ordinal;
        return ordinal < bb.n_map ? bb.map[ordinal] : 0xFFFFFFFFu;   // push_dummy_index (:703-705)
    };
    if (bb.mode == 1u) {   // storage: (offset, point, spot, rect | probes, volumes, decals, 0) per cluster (:636-652)
        for (uint32_t c = tid; c < nc; c += nth) {
            const uint32_t len = off[c + 1] - off[c];
            if (bb.kind == nullptr) {
                reinterpret_cast<uint4 *>(oc)[c * 2] = make_uint4(off[c], len, 0u, 0u);
                reinterpret_cast<uint4 *>(oc)[c * 2 + 1] = make_uint4(0u, 0u, 0u, 0u);
                continue;
            }
            // ObjectsInClusterCpu::add_* (bevy_light/src/cluster/mod.rs:478-512): one counter per kind; the entries that did
            // not fit max_cluster_indices count as point lights
            uint32_t n_kind[6] = {0u, 0u, 0u, 0u, 0u, 0u};
            for (uint32_t i = off[c]; i < min(off[c + 1], avail); ++i) ++n_kind[min((uint32_t)bb.kind[idx[i]], 5u)];
            const uint32_t objects = n_kind[kKindRect] + n_kind[kKindReflectionProbe] + n_kind[kKindIrradianceVolume] + n_kind[kKindDecal];
            reinterpret_cast<uint4 *>(oc)[c * 2] = make_uint4(off[c], len - objects, 0u, n_kind[kKindRect]);
            reinterpret_cast<uint4 *>(oc)[c * 2 + 1] = make_uint4(n_kind[kKindReflectionProbe], n_kind[kKindIrradianceVolume], n_kind[kKindDecal], 0u);
        }
        for (uint32_t i = tid; i < avail; i += nth) il[i] = gpu_index(idx[i]);
        if (tid == 0) { bb.count[v * 2] = nc; bb.count[v * 2 + 1] = avail; }
    } else {               // uniform: packed offset|counts words and 8-bit indices, truncated at MAX_INDICES (:505-514)
        const uint32_t n_ind = min(avail, kMaxIndices);
        // the record loop breaks at the first Light with n_indices >= MAX_INDICES: headers exist exactly for the
        // clusters whose offset is <= MAX_INDICES (offsets are monotone)
        for (uint32_t c = tid; c < kUniformWords; c += nth) {
            uint32_t w = 0;
            if (c < nc && off[c] <= kMaxIndices)
                w = ((off[c] & ((1u << (32u - 2u * kCountSize)) - 1u)) << (2u * kCountSize)) |
                    (((off[c + 1] - off[c]) & ((1u << kCountSize) - 1u)) << kCountSize);   // pack_offset_and_counts (:855-859)
            oc[c] = w;
        }
        for (uint32_t w = tid; w < kUniformWords; w += nth) {
            uint32_t word = 0;
#pragma unroll
            for (uint32_t s = 0; s < 4; ++s) { const uint32_t i = w * 4 + s; if (i < n_ind) word |= gpu_index(idx[i]) << (8u * s); }   // (:676-686)
            il[w] = word;
        }
        if (tid == 0) {
            uint32_t lo = 0, hi = nc;   // number of clusters with off[c] <= kMaxIndices
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (off[mid] <= kMaxIndices) lo = mid + 1; else hi = mid; }
            bb.count[v * 2] = lo; bb.count[v * 2 + 1] = n_ind;
        }
    }
}

// ------------------------------------------------------------------------------------------
// pack / unpack kernels for the C ABI's AoS <-> device SoA conversion
// ------------------------------------------------------------------------------------------
__global__ void k_unpack_trs(Rows R, uint32_t first, uint32_t count, const float *__restrict__ src, int mark_only) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t row = first + i;
    if (!mark_only) {
        const float *t = src + (size_t)i * 10;
        R.trsA[row] = make_float4(t[0], t[1], t[2], t[7]);
        R.trsB[row] = make_float4(t[3], t[4], t[5], t[6]);
        R.trsC[row] = make_float2(t[8], t[9]);
    }
    R.flags[row] = (uint8_t)(R.flags[row] | F_TCHANGED);
}
__global__ void k_scatter_trs(Rows R, uint32_t count, const uint32_t *__restrict__ rows, const float *__restrict__ src) {
    asm volatile("griddepcontrol.wait;" ::: "memory");   // PDL: the previous frame's tile pass still reads these columns
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t row = rows[i];
    if (row >= R.n) return;
    const float *t = src + (size_t)i * 10;
    R.trsA[row] = make_float4(t[0], t[1], t[2], t[7]);
    R.trsB[row] = make_float4(t[3], t[4], t[5], t[6]);
    R.trsC[row] = make_float2(t[8], t[9]);
    R.flags[row] = (uint8_t)(R.flags[row] | F_TCHANGED);
}
__global__ void k_unpack_gt(Rows R, uint32_t first, uint32_t count, const float *__restrict__ src) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const float *g = src + (size_t)i * 12;   // X.xyz Y.xyz Z.xyz T.xyz
    const uint32_t row = first + i;
    R.gt0[row] = make_float4(g[0], g[3], g[6], g[9]);
    R.gt1[row] = make_float4(g[1], g[4], g[7], g[10]);
    R.gt2[row] = make_float4(g[2], g[5], g[8], g[11]);
}
__global__ void k_pack_gt(Rows R, uint32_t first, uint32_t count, float *__restrict__ dst, uint32_t stride) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t row = first + i;
    const float4 a = R.gt0[row], b = R.gt1[row], c = R.gt2[row];
    float *g = dst + (size_t)i * stride;
    if (stride == 12) {
        g[0] = a.x; g[1] = b.x; g[2] = c.x; g[3] = a.y; g[4] = b.y; g[5] = c.y;
        g[6] = a.z; g[7] = b.z; g[8] = c.z; g[9] = a.w; g[10] = b.w; g[11] = c.w;
    } else {   // glam Affine3A: four 16-byte Vec3A lanes
        g[0] = a.x; g[1] = b.x; g[2] = c.x; g[3] = 0.0f; g[4] = a.y; g[5] = b.y; g[6] = c.y; g[7] = 0.0f;
        g[8] = a.z; g[9] = b.z; g[10] = c.z; g[11] = 0.0f; g[12] = a.w; g[13] = b.w; g[14] = c.w; g[15] = 0.0f;
    }
}
__global__ void k_unpack_bounds(Rows R, uint32_t first, uint32_t count, const float *__restrict__ bounds,
                                const uint8_t *__restrict__ flags, const uint8_t *__restrict__ cls, uint8_t *__restrict__ cls_col) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t row = first + i;
    const float *b = bounds + (size_t)i * 6;
    R.bndA[row] = make_float4(b[0], b[1], b[2], b[3]);
    R.bndB[row] = make_float2(b[4], b[5]);
    R.flags[row] = (uint8_t)((flags[i] & 0x7Fu) | (R.flags[row] & F_TCHANGED));
    R.state[row] = (uint8_t)((R.state[row] & ~S_HAS_CLASS) | (cls[i] ? S_HAS_CLASS : 0u));
    cls_col[row] = cls[i];
}
__global__ void k_unpack_vv(Rows R, uint32_t first, uint32_t count, const uint8_t *__restrict__ vv) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t row = first + i;
    R.state[row] = (uint8_t)((R.state[row] & ~S_VV) | (vv[i] & S_VV));
}
// ------------------------------------------------------------------------------------------
// SURVEY 8(f) N4: visibility_propagate_system (crates/bevy_camera/src/visibility/mod.rs:638-729) as a level walk
// over the transform plan's tiles.  The reference is change-driven; this computes the state it converges to:
// Visible -> true, Hidden -> false, Inherited -> the parent's InheritedVisibility, or true when there is no parent or
// the parent lacks the components (:655-659).  Writes only where the value differs (:667) and flags those rows.
// ------------------------------------------------------------------------------------------
constexpr uint32_t V_HIDDEN = 1u, V_VISIBLE = 2u, V_NO_COMPONENTS = 4u;
__global__ void __launch_bounds__(kTileRows)
k_visibility_propagate(Rows R, const Tile *__restrict__ tiles, const uint8_t *__restrict__ vis, uint8_t *__restrict__ changed) {
    __shared__ uint8_t s_inh[kTileRows];   // 0 / 1, or 2 = the row lacks the components
    const Tile tile = tiles[blockIdx.x];
    const uint32_t lr = threadIdx.x, row = tile.base + lr;
    const bool active = lr < tile.n_rows;
    const uint32_t topo = active ? R.topo[row] : 0u, f = active ? R.flags[row] : 0u, v = active ? vis[row] : V_NO_COMPONENTS;
    const uint32_t my_level = active ? ((topo >> 9) & 0x1FFu) : 0xFFFFFFFFu;
    uint32_t inh = 0;
    for (uint32_t lvl = 0; lvl < tile.n_levels; ++lvl) {
        if (lvl) __syncthreads();
        if (my_level == lvl) {
            uint32_t parent_inh = 1u;   // no parent (root) or a parent outside the hierarchy the library knows
            if (topo & T_EXT_PARENT) {
                const uint32_t pr = R.parent[row];
                if (!(vis[pr] & V_NO_COMPONENTS)) parent_inh = R.flags[pr] & F_INHERITED;   // settled by an earlier pass
            } else if (!(topo & (T_ROOT | T_DETACHED))) {
                const uint32_t p = s_inh[topo & 0x1FFu];
                parent_inh = p == 2u ? 1u : p;
            }
            inh = (v & 3u) == V_VISIBLE ? 1u : (v & 3u) == V_HIDDEN ? 0u : parent_inh;
            s_inh[lr] = (v & V_NO_COMPONENTS) ? 2u : (uint8_t)inh;
        }
    }
    if (active) {
        const bool write = !(v & V_NO_COMPONENTS) && (f & F_INHERITED) != inh;
        if (write) R.flags[row] = (uint8_t)(f ^ F_INHERITED);
        changed[row] = write ? 1 : 0;
    }
}
// out[0..count) = InheritedVisibility, out[count..2count) = written by the last k_visibility_propagate
__global__ void k_pack_inherited(Rows R, uint32_t first, uint32_t count, const uint8_t *__restrict__ changed, uint8_t *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    out[i] = (uint8_t)(R.flags[first + i] & F_INHERITED);
    out[count + i] = changed ? changed[first + i] : 0;
}
// VisibleEntityRanges::entities values: 0 (= no entry) unless the row is in check_visibility_ranges' query
__global__ void k_pack_ranges(Rows R, uint32_t first, uint32_t count, uint32_t *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t f = R.flags[first + i];
    out[i] = ((f & F_RANGE) && !(f & F_NO_CPU_CULL)) ? R.range[first + i] : 0u;
}
__global__ void k_unpack_range_params(float2 *__restrict__ se, uint8_t *__restrict__ ua, uint32_t first, uint32_t count,
                                      const float *__restrict__ src_se, const uint8_t *__restrict__ src_ua) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    se[first + i] = make_float2(src_se[i * 2], src_se[i * 2 + 1]);
    ua[first + i] = src_ua[i];
}

// out[0..count) = vv byte, out[count..2count) = changed byte selected by `changed_bit`
__global__ void k_pack_state(Rows R, uint32_t first, uint32_t count, uint8_t *__restrict__ out, uint32_t changed_bit) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t s = R.state[first + i];
    out[i] = (uint8_t)(s & S_VV);
    out[count + i] = (s & changed_bit) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
static inline unsigned cdiv(unsigned a, unsigned b) { return (a + b - 1) / b; }
// kernel launches issued by this library since load (bench.py reports the difference over its timed region)
static unsigned long long g_launches = 0;
unsigned long long kernel_launch_count() { return g_launches; }

// Function attributes (dynamic shared memory size, cluster size) are per DEVICE: a process that drives several GPUs
// (b200vis_p2p_link) must set them on each.  Returns true the first time it is called for (this call site, current device).
static bool first_call_on_device(unsigned long long &seen) {
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long bit = 1ull << (dev & 63);
    if (seen & bit) return false;
    seen |= bit;
    return true;
}
static int g_tile_kernel = -1;   // 5 lean (default: TMA-staged, bookkeeping thread, top levels in registers, rolled view loop), 0 classic (one tile per CTA, LDG), 1 kernel 1b (persistent TMA-staged CTA per tile), 2 warp per tile, 3 TMA + scout warp, 4 TMA flow (no inter-tile barrier)
static int tile_kernel_choice() {
    if (g_tile_kernel < 0) {
        const char *e = getenv("B200VIS_TILE_KERNEL");
        g_tile_kernel = (e && e[0] == 'c') ? 0 : (e && e[0] == 'w') ? 2 : (e && e[0] == 's') ? 3 : (e && e[0] == 'f') ? 4 : (e && e[0] == 't') ? 1 : 5;      // default: lean (kernel 1L); tma = kernel 1b
    }
    return g_tile_kernel;
}
static int lean_ctas_per_sm() {       // B200VIS_LEAN_CTAS = 4 | 5 | 6 resident CTAs per SM of the lean kernel
    static int n = 0;
    if (!n) { const char *e = getenv("B200VIS_LEAN_CTAS"); n = (e && (atoi(e) == 5 || atoi(e) == 6)) ? atoi(e) : 4; }
    return n;
}
static bool lean_pipe() {       // B200VIS_LEAN_PIPE=1: the CTA's warps are not held together at tile boundaries (measured slower: DESIGN.md section 7)
    static int v = -1;
    if (v < 0) { const char *e = getenv("B200VIS_LEAN_PIPE"); v = (e && atoi(e) == 1) ? 1 : 0; }
    return v != 0;
}
bool tile_kernel_is_tma() { return tile_kernel_choice() == 1 || tile_kernel_choice() == 3 || tile_kernel_choice() == 4 || tile_kernel_choice() == 5; }
bool tile_kernel_publishes_light_snapshot() { return tile_kernel_choice() != 0; }
template <bool C, bool S, int MINB, bool PIPE>
static void launch_warp(cudaStream_t st, const Rows &R, const WarpTile *tiles, const uint8_t *sched, uint32_t n_tiles, const CullViews &cvw,
                        const VisibleBufs &vb, DevStats *stats, uint32_t static_opt, uint32_t parity, uint32_t *counter) {
    constexpr size_t smem = (kTileRows / 32) * sizeof(WarpSmem);
    static int grid = 0, dynamic = 0;
    static unsigned long long seen = 0;
    if (first_call_on_device(seen)) {
        cudaFuncSetAttribute(k_tile_warp<C, S, MINB, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int dev = 0, sms = 0, per_sm = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tile_warp<C, S, MINB, PIPE>, kTileRows, smem);
        if (per_sm > MINB) per_sm = MINB;
        grid = sms * (per_sm > 0 ? per_sm : 1);
        const char *d = getenv("B200VIS_WARP_DYNAMIC");   // tiles handed out by an atomic counter instead of a fixed stride
        dynamic = (d && atoi(d)) ? 1 : 0;
    }
    const uint32_t need = (n_tiles + (kTileRows / 32) - 1) / (kTileRows / 32);
    const uint32_t g = need < (uint32_t)grid ? need : (uint32_t)grid;
    uint32_t *ctr = nullptr;
    if (dynamic && counter != nullptr) { cudaMemsetAsync(counter, 0, 4, st); ctr = counter; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g); cfg.blockDim = dim3(kTileRows); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ++g_launches; cudaLaunchKernelEx(&cfg, k_tile_warp<C, S, MINB, PIPE>, R, tiles, sched, n_tiles, cvw, vb, stats, static_opt, parity, ctr);
}
template <int MINB, bool PIPE>
static void launch_tile_warp_m(cudaStream_t st, const Rows &R, const WarpTile *tiles, const uint8_t *sched, uint32_t n_tiles, const CullViews &cvw,
                               const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity, uint32_t *counter) {
    const bool cull = stages & 2u;
    const bool simple = R.layers == nullptr && R.layers_ext == nullptr && R.range == nullptr && R.rank == nullptr;
    if (cull) { if (simple) launch_warp<true, true, MINB, PIPE>(st, R, tiles, sched, n_tiles, cvw, vb, stats, static_opt, parity, counter);
                else launch_warp<true, false, MINB, PIPE>(st, R, tiles, sched, n_tiles, cvw, vb, stats, static_opt, parity, counter); }
    else launch_warp<false, true, MINB, PIPE>(st, R, tiles, sched, n_tiles, cvw, vb, stats, static_opt, parity, counter);
}
void launch_tile_warp(cudaStream_t st, const Rows &R, const WarpTile *tiles, const uint8_t *sched, uint32_t n_tiles, const CullViews &cvw,
                      const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity, uint32_t *counter) {
    if (n_tiles == 0) return;
    // B200VIS_WARP_VARIANT = <CTAs per SM><p|n>: 4 = 32 warps per SM at 64 registers, 3 = 24 at 80, 2 = 16 at 128;
    // p = next chunk loaded into registers during the cull, n = only prefetched into L2
    static int variant = -1;
    if (variant < 0) {
        const char *e = getenv("B200VIS_WARP_VARIANT");
        const int b = (e && e[0] >= '2' && e[0] <= '4') ? e[0] - '0' : 3;
        const int pipe = (e && e[0] && e[1] == 'n') ? 0 : 1;
        variant = b * 2 + pipe;
    }
#define B200VIS_WARP_CASE(B, P) case (B) * 2 + (P): launch_tile_warp_m<B, P != 0>(st, R, tiles, sched, n_tiles, cvw, vb, stats, stages, static_opt, parity, counter); break
    switch (variant) {
        B200VIS_WARP_CASE(4, 1); B200VIS_WARP_CASE(4, 0); B200VIS_WARP_CASE(3, 1); B200VIS_WARP_CASE(3, 0);
        B200VIS_WARP_CASE(2, 1); B200VIS_WARP_CASE(2, 0);
    }
#undef B200VIS_WARP_CASE
}
bool tile_kernel_is_warp() { return tile_kernel_choice() == 2; }
template <bool C, bool S, int MINB>
static void launch_scout(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw,
                         const VisibleBufs &vb, DevStats *stats, uint32_t static_opt, uint32_t parity) {
    static int grid = 0, tiles_per_cta = 0;
    static unsigned long long seen = 0;
    if (first_call_on_device(seen)) {
        cudaFuncSetAttribute(k_propagate_cull_scout<C, S, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScoutSmem));
        int dev = 0, sms = 0, per_sm = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate_cull_scout<C, S, MINB>, kScoutThreads, sizeof(ScoutSmem));
        grid = sms * (per_sm > 0 ? per_sm : 1);    // persistent: one CTA per resident slot
        // B200VIS_SCOUT_TILES_PER_CTA=k bounds the tiles one CTA walks (0 = fully persistent, the default: the scout's
        // one-tile lead pays off over a run of tiles; the first tile of every CTA has none)
        const char *e = getenv("B200VIS_SCOUT_TILES_PER_CTA");
        tiles_per_cta = e ? atoi(e) : 0;
    }
    uint32_t g = n_tiles < (uint32_t)grid ? n_tiles : (uint32_t)grid;
    if (tiles_per_cta > 0) {
        uint32_t want = (n_tiles + tiles_per_cta - 1) / tiles_per_cta;
        want = ((want + (uint32_t)grid - 1) / (uint32_t)grid) * (uint32_t)grid;      // whole waves of resident CTAs
        if (want > n_tiles) want = n_tiles;
        if (want > g) g = want;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g); cfg.blockDim = dim3(kScoutThreads); cfg.dynamicSmemBytes = sizeof(ScoutSmem); cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ++g_launches; cudaLaunchKernelEx(&cfg, k_propagate_cull_scout<C, S, MINB>, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity);
}
template <int MINB>
static void launch_scout_m(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw, const VisibleBufs &vb,
                           DevStats *stats, bool cull, bool simple, uint32_t static_opt, uint32_t parity) {
    if (cull) { if (simple) launch_scout<true, true, MINB>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity);
                else launch_scout<true, false, MINB>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity); }
    else launch_scout<false, true, MINB>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity);
}
template <bool P, bool C, bool S, int KIND>      // KIND: 0 kernel 1b, 1 flow, 4 / 5 / 6 lean with that many CTAs per SM, 7 lean with drifting warps (PIPE)
static void launch_tma(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw,
                       const VisibleBufs &vb, DevStats *stats, uint32_t static_opt, uint32_t parity, uint32_t *ticket, uint32_t *ticket_base) {
    static int grid = 0;
    static unsigned long long seen = 0;
    constexpr bool FLOW = KIND == 1;
    constexpr size_t smem = (KIND == 4 || KIND == 7) ? sizeof(LeanSmem<true>) : KIND >= 5 ? sizeof(LeanSmem<false>) : sizeof(TmaSmem);
    auto with_kernel = [&](auto &&fn) {
        if constexpr (KIND == 1) fn(k_propagate_cull_flow<P, C, S>);
        else if constexpr (KIND == 4) fn(k_propagate_cull_lean<P, C, S, 4>);
        else if constexpr (KIND == 5) fn(k_propagate_cull_lean<P, C, S, 5>);
        else if constexpr (KIND == 6) fn(k_propagate_cull_lean<P, C, S, 6>);
        else if constexpr (KIND == 7) fn(k_propagate_cull_lean<P, C, S, 4, P && C>);
        else fn(k_propagate_cull_tma<P, C, S>);
    };
    if (first_call_on_device(seen)) {
        with_kernel([&](auto kern) {
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            int dev = 0, sms = 0, per_sm = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kTileRows, smem);
            grid = sms * (per_sm > 0 ? per_sm : 1);    // persistent: one CTA per resident slot
        });
    }
    uint32_t g = n_tiles < (uint32_t)grid ? n_tiles : (uint32_t)grid;
    // B200VIS_TILES_PER_CTA=k (default 0 = fully persistent, measured best in round 2; round 1 used 2) bounds the tiles one CTA processes (grid = n_tiles / k):
    // CTAs then retire continuously, which lets the (higher priority) tail kernels of the previous frame and the
    // all-gather slip in between instead of waiting for the whole persistent grid to drain
    static int tiles_per_cta = -1;
    if (tiles_per_cta < 0) { const char *e = getenv("B200VIS_TILES_PER_CTA"); tiles_per_cta = e ? atoi(e) : 0; }
    if (tiles_per_cta > 0) {
        // round the grid up to whole waves of resident CTAs: the surplus CTAs then take one tile fewer, so the last
        // wave is made of short CTAs instead of a few full-length ones running on a mostly idle chip
        uint32_t want = (n_tiles + tiles_per_cta - 1) / tiles_per_cta;
        static int balance = -1;
        if (balance < 0) { const char *e = getenv("B200VIS_BALANCE_WAVES"); balance = e ? atoi(e) : 1; }
        if (balance) want = ((want + (uint32_t)grid - 1) / (uint32_t)grid) * (uint32_t)grid;
        if (want > n_tiles) want = n_tiles;
        if (want > g) g = want;
    }
    // programmatic dependent launch: this kernel's CTAs may become resident (barrier init, parameter loads) while the
    // previous kernel in the stream drains; griddepcontrol.wait in the kernel orders the actual data accesses
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g); cfg.blockDim = dim3(kTileRows); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    // dynamic tile hand-out (fully persistent grids of the default kernel; B200VIS_TILE_HANDOUT=static keeps the fixed stride)
    static int dynamic = -1;
    if (dynamic < 0) { const char *e = getenv("B200VIS_TILE_HANDOUT"); dynamic = (e && e[0] == 's') ? 0 : 1; }
    uint32_t *tk = nullptr, base = 0;
    if (!FLOW && dynamic && tiles_per_cta == 0 && ticket && ticket_base) { tk = ticket; base = *ticket_base; *ticket_base += n_tiles; }
    ++g_launches;
    with_kernel([&](auto kern) {
        if constexpr (KIND >= 4) {
            static int flip = -1;     // B200VIS_LEAN_WARP_FLIP=1 reverses the CTA's warp order (no measurable effect: DESIGN.md section 7)
            if (flip < 0) { const char *e = getenv("B200VIS_LEAN_WARP_FLIP"); flip = (e && atoi(e) == 1) ? 0xE0 : 0; }
            static int probe = -1;    // B200VIS_LEAN_PROBE: timing probes, wrong results (tools/ only)
            if (probe < 0) { const char *e = getenv("B200VIS_LEAN_PROBE"); probe = e ? atoi(e) : 0; }
            cudaLaunchKernelEx(&cfg, kern, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, tk, base, (uint32_t)flip | ((uint32_t)probe << 8));
        } else {
            cudaLaunchKernelEx(&cfg, kern, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, tk, base);
        }
    });
}
// tiles of <= 32 rows (the tops of split deep tiles): the classic kernel with one warp per tile, 16 CTAs per SM
void launch_propagate_cull_small(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw,
                                 const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity) {
    if (n_tiles == 0) return;
    const bool prop = stages & 1u, cull = stages & 2u;
    const bool simple = R.layers == nullptr && R.layers_ext == nullptr && R.range == nullptr && R.rank == nullptr;
#define B200VIS_LAUNCH_SMALL(P, C, S) ++g_launches, k_propagate_cull<P, C, S><<<n_tiles, 32, 0, st>>>(R, tiles, cvw, vb, stats, static_opt, parity)
    if (prop && cull) { if (simple) B200VIS_LAUNCH_SMALL(true, true, true); else B200VIS_LAUNCH_SMALL(true, true, false); }
    else if (prop) B200VIS_LAUNCH_SMALL(true, false, true);
    else if (cull) { if (simple) B200VIS_LAUNCH_SMALL(false, true, true); else B200VIS_LAUNCH_SMALL(false, true, false); }
#undef B200VIS_LAUNCH_SMALL
}
void launch_propagate_cull(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw,
                           const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity,
                           uint32_t *ticket, uint32_t *ticket_base, bool named_levels_only) {
    if (n_tiles == 0) return;
    const bool prop = stages & 1u, cull = stages & 2u;
    const bool simple = R.layers == nullptr && R.layers_ext == nullptr && R.range == nullptr && R.rank == nullptr;
    if (tile_kernel_choice() == 3 && prop) {       // TMA-staged tiles + a scout warp one tile ahead (B200VIS_TILE_KERNEL=scout)
        static int per_sm = 0;      // 3 CTAs per SM at 64 registers (default) or 2 at ~100
        if (!per_sm) { const char *e = getenv("B200VIS_SCOUT_CTAS_PER_SM"); per_sm = (e && atoi(e) == 2) ? 2 : 3; }
        if (per_sm == 2) launch_scout_m<2>(st, R, tiles, n_tiles, cvw, vb, stats, cull, simple, static_opt, parity);
        else launch_scout_m<3>(st, R, tiles, n_tiles, cvw, vb, stats, cull, simple, static_opt, parity);
        return;
    }
    if (tile_kernel_is_tma()) {
#define B200VIS_LAUNCH_TMA(P, C, S) do { if (tile_kernel_choice() == 4) launch_tma<P, C, S, 1>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, ticket, ticket_base); \
                                         else if (tile_kernel_choice() == 5 && lean_ctas_per_sm() == 4 && (P) && (C) && named_levels_only && lean_pipe()) launch_tma<P, C, S, 7>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, ticket, ticket_base); \
                                         else if (tile_kernel_choice() == 5 && lean_ctas_per_sm() == 4) launch_tma<P, C, S, 4>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, ticket, ticket_base); \
                                         else if (tile_kernel_choice() == 5 && lean_ctas_per_sm() == 6) launch_tma<P, C, S, 6>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, ticket, ticket_base); \
                                         else if (tile_kernel_choice() == 5) launch_tma<P, C, S, 5>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, ticket, ticket_base); \
                                         else launch_tma<P, C, S, 0>(st, R, tiles, n_tiles, cvw, vb, stats, static_opt, parity, ticket, ticket_base); } while (0)
        if (prop && cull) { if (simple) B200VIS_LAUNCH_TMA(true, true, true); else B200VIS_LAUNCH_TMA(true, true, false); }
        else if (prop) B200VIS_LAUNCH_TMA(true, false, true);
        else if (cull) { if (simple) B200VIS_LAUNCH_TMA(false, true, true); else B200VIS_LAUNCH_TMA(false, true, false); }
#undef B200VIS_LAUNCH_TMA
        return;
    }
#define B200VIS_LAUNCH(P, C, S) ++g_launches, k_propagate_cull<P, C, S><<<n_tiles, kTileRows, 0, st>>>(R, tiles, cvw, vb, stats, static_opt, parity)
    if (prop && cull) { if (simple) B200VIS_LAUNCH(true, true, true); else B200VIS_LAUNCH(true, true, false); }
    else if (prop) B200VIS_LAUNCH(true, false, true);
    else if (cull) { if (simple) B200VIS_LAUNCH(false, true, true); else B200VIS_LAUNCH(false, true, false); }
#undef B200VIS_LAUNCH
}
void launch_cull(cudaStream_t st, const Rows &R, const CullViews &cvw, const VisibleBufs &vb, DevStats *stats, uint32_t parity) {
    if (!R.n) return;
    const bool simple = R.layers == nullptr && R.layers_ext == nullptr && R.range == nullptr && R.rank == nullptr;
    if (simple) { ++g_launches; k_cull<true><<<cdiv(R.n, 256), 256, 0, st>>>(R, cvw, vb, stats, parity); }
    else { ++g_launches; k_cull<false><<<cdiv(R.n, 256), 256, 0, st>>>(R, cvw, vb, stats, parity); }
}
void launch_mark_dirty_global(cudaStream_t st, const Rows &R) {
    if (R.n) { ++g_launches; k_mark_dirty_global<<<cdiv(R.n, 256), 256, 0, st>>>(R); }
}
void launch_expand_visible(cudaStream_t st, const VisibleBufs &vb, const DiffBufs &db, const uint32_t *row_of_rank, const FrameConsts *fc,
                           DevStats *stats, uint32_t parity, uint32_t n_rows, uint32_t max_views) {
    if (vb.n_chunks == 0) return;
    ++g_launches; k_expand_visible<<<dim3(vb.n_chunks, max_views), kChunkWords, 0, st>>>(vb, db, row_of_rank, fc, stats, parity, n_rows);
    if (db.prev != nullptr) { ++g_launches; k_emit_visible_diff<<<dim3(vb.n_chunks, max_views), kChunkWords, 0, st>>>(vb, db, row_of_rank, fc); }
}
void launch_publish_visible_diff(cudaStream_t st, const VisibleBufs &vb, const DiffBufs &db, uint32_t *host_rows, uint32_t host_stride,
                                 uint32_t *host_counts, uint32_t n_views, uint32_t max_views) {
    if (!n_views || db.prev == nullptr) return;
    ++g_launches; k_publish_visible_diff<<<dim3(32, n_views, 2), 256, 0, st>>>(db, vb.list_stride, host_rows, host_stride, host_counts, n_views, max_views);
}
void launch_cluster_assign(cudaStream_t st, const Rows &R, const Lights &L, const FrameConsts *fc, const ClusterBufs &cb,
                           DevStats *stats, uint32_t max_views) {
    if (L.n == 0) return;
    ++g_launches; k_cluster_assign<<<dim3(cdiv(L.n, 8), max_views), 256, 0, st>>>(R, L, fc, cb, stats);
}
// assign + lists of every view in one launch (single GPU): thread-block clusters of 8 (16 beyond ~3200 lights) CTAs per view
// Can the one-launch cluster stage hold `n_lights` mask bits per cluster in a thread-block cluster's shared memory?
bool cluster_fused_fits(uint32_t n_lights) {
    const char *e = getenv("B200VIS_CLUSTER_KERNEL");
    if (e && e[0] == 's') return false;
    const size_t words = (n_lights + 31u) / 32u;
    return words * (kMaxClusters / 16) * 4 <= 200u * 1024u;
}
bool launch_cluster_fused(cudaStream_t st, const Rows &R, const Lights &L, const FrameConsts *fc, const ClusterBufs &cb,
                          DevStats *stats, uint32_t max_views) {
    static int enabled = -1, nrank_env = 0;
    static unsigned long long seen = 0;
    if (enabled < 0) {
        const char *e = getenv("B200VIS_CLUSTER_KERNEL");
        enabled = (e && e[0] == 's') ? 0 : 1;                 // "split": the assign / lists / clear kernels
        const char *r = getenv("B200VIS_CLUSTER_CTAS");
        nrank_env = r ? atoi(r) : 0;
    }
    if (first_call_on_device(seen)) {
        cudaFuncSetAttribute(k_cluster_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_cluster_fused, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    }
    if (!enabled) return false;
    const uint32_t words = (L.n + 31u) / 32u;
    uint32_t nrank = (nrank_env == 2 || nrank_env == 4 || nrank_env == 8 || nrank_env == 16) ? (uint32_t)nrank_env : 8u;
    size_t smem = (size_t)words * (kMaxClusters / nrank) * 4;
    if (smem > 200u * 1024u) { nrank = 16; smem = (size_t)words * (kMaxClusters / nrank) * 4; }
    if (smem > 200u * 1024u) return false;                    // more lights than the distributed matrix can hold: split path
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nrank, max_views); cfg.blockDim = dim3(kFusedThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = nrank; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ++g_launches; return cudaLaunchKernelEx(&cfg, k_cluster_fused, R, L, fc, cb, stats) == cudaSuccess;
}
void launch_publish_visible(cudaStream_t st, const VisibleBufs &vb, const DevStats *stats, uint32_t *host_rows, uint32_t host_stride,
                            uint32_t n_rows, uint32_t n_views, uint8_t *host_classes) {
    if (!n_views || !n_rows) return;
    ++g_launches; k_publish_visible<<<dim3(min(cdiv(n_rows, 256), 296u), n_views), 256, 0, st>>>(vb.lists, vb.list_stride, stats, host_rows, host_stride, n_views, vb.classes, host_classes);
}
void launch_publish_clusters(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, uint32_t *host_offsets, uint32_t *host_indices,
                             uint32_t host_cap, const DevStats *stats, uint32_t *host_stats, uint32_t changed_slot, uint32_t frame, uint32_t max_views) {
    ++g_launches; k_publish_clusters<<<dim3(kMaxClusters / 256 + 1, max_views), 256, 0, st>>>(fc, cb.offsets, cb.indices, cb.index_cap, host_offsets, host_indices,
                                                                                host_cap, stats, host_stats, changed_slot, frame);
}
void launch_shadow_cull(cudaStream_t st, const Rows &R, const ShadowBufs &sb, const uint32_t *view_sets, uint32_t n_views,
                        uint32_t n_words, uint32_t n_chunks, uint32_t words_stride, uint32_t chunks_stride, DevStats *stats, uint32_t changed_slot) {
    if (!sb.n_lights || !R.n) return;
    ++g_launches; k_shadow_select<<<cdiv(sb.n_lights, 128), 128, 0, st>>>(sb, R.rank, view_sets, words_stride, n_views);
    ++g_launches; k_shadow_cull<<<cdiv(R.n, 256), 256, 0, st>>>(R, sb, words_stride, chunks_stride, stats, changed_slot);
    ++g_launches; k_expand_shadow<<<dim3(n_chunks, sb.n_lights), kChunkWords, 0, st>>>(sb, n_words, n_chunks, words_stride, chunks_stride, R.row_of_rank);
}
void launch_pack_cluster_bindings(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, const BindingBufs &bb, uint32_t max_views) {
    if (bb.mode) { ++g_launches; k_pack_cluster_bindings<<<dim3(16, max_views), 256, 0, st>>>(fc, cb, bb); }
}
void launch_tag_lights(cudaStream_t st, const Rows &R, const Lights &L, uint32_t *light_ord, uint32_t *all_tagged) {
    if (L.n) { ++g_launches; k_tag_lights<<<cdiv(L.n, 128), 128, 0, st>>>(R, L, light_ord, all_tagged); }
}
void launch_snapshot_lights(cudaStream_t st, const Rows &R, const Lights &L, float4 *snap) {
    if (L.n) { ++g_launches; k_snapshot_lights<<<cdiv(L.n, 128), 128, 0, st>>>(R, L, snap); }
}
void launch_snapshot_objects(cudaStream_t st, const Rows &R, const ClusterObjects &O, float4 *snap, float *range) {
    if (O.n) { ++g_launches; k_snapshot_objects<<<cdiv(O.n, 128), 128, 0, st>>>(R, O, snap, range); }
}
void launch_writeback_columns(cudaStream_t st, const Rows &R, float *host_gt, uint32_t stride, uint32_t *host_gt_bits, uint8_t *host_vv,
                              uint32_t *host_vv_bits, uint8_t *vv_shadow) {
    if (!R.n) return;
    const unsigned groups = cdiv(R.n, 128), grid = groups < 8u * 1184u ? cdiv(groups, 8) : 1184u;
    if (stride == 16) { ++g_launches; k_writeback_columns<16><<<grid, 256, 0, st>>>(R, host_gt, host_gt_bits, host_vv, host_vv_bits, vv_shadow); }
    else { ++g_launches; k_writeback_columns<12><<<grid, 256, 0, st>>>(R, host_gt, host_gt_bits, host_vv, host_vv_bits, vv_shadow); }
}
void launch_record_push(cudaStream_t st, const uint32_t *block, uint32_t block_words, const ClusterBufs &cb) {
    ++g_launches; k_record_push<<<cb.world, 256, 0, st>>>(block, block_words, cb);
}
void launch_slab_push(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, uint32_t *done, uint32_t max_views) {
    ++g_launches; k_slab_push<<<dim3(8, max_views), 256, 0, st>>>(fc, cb, done);
}
void launch_cluster_lists(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, DevStats *stats, uint32_t max_views) {
    ++g_launches; k_cluster_lists<<<dim3(kListBlocks, max_views), 1024, 0, st>>>(fc, cb, stats);
    ++g_launches; k_cluster_clear<<<dim3(kMaxClusters / 256, max_views), 256, 0, st>>>(fc, cb);
}
void launch_unpack_trs(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const float *src, int mark_only) {
    if (count) { ++g_launches; k_unpack_trs<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, src, mark_only); }
}
void launch_scatter_trs(cudaStream_t st, const Rows &R, uint32_t count, const uint32_t *rows, const float *src) {
    if (!count) return;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cdiv(count, 256)); cfg.blockDim = dim3(256); cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ++g_launches; cudaLaunchKernelEx(&cfg, k_scatter_trs, R, count, rows, src);
}
void launch_unpack_gt(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const float *src) {
    if (count) { ++g_launches; k_unpack_gt<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, src); }
}
void launch_pack_gt(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, float *dst, uint32_t stride) {
    if (count) { ++g_launches; k_pack_gt<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, dst, stride); }
}
void launch_unpack_bounds(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const float *bounds,
                          const uint8_t *flags, const uint8_t *cls, uint8_t *cls_col) {
    if (count) { ++g_launches; k_unpack_bounds<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, bounds, flags, cls, cls_col); }
}
void launch_unpack_vv(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const uint8_t *vv) {
    if (count) { ++g_launches; k_unpack_vv<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, vv); }
}
void launch_visibility_propagate(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const uint8_t *vis, uint8_t *changed) {
    if (n_tiles) { ++g_launches; k_visibility_propagate<<<n_tiles, kTileRows, 0, st>>>(R, tiles, vis, changed); }
}
void launch_pack_inherited(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const uint8_t *changed, uint8_t *out) {
    if (count) { ++g_launches; k_pack_inherited<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, changed, out); }
}
void launch_pack_ranges(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, uint32_t *out) {
    if (count) { ++g_launches; k_pack_ranges<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, out); }
}
void launch_unpack_range_params(cudaStream_t st, float2 *se, uint8_t *ua, uint32_t first, uint32_t count, const float *src_se, const uint8_t *src_ua) {
    if (count) { ++g_launches; k_unpack_range_params<<<cdiv(count, 256), 256, 0, st>>>(se, ua, first, count, src_se, src_ua); }
}
void launch_pack_state(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, uint8_t *out, uint32_t changed_bit) {
    if (count) { ++g_launches; k_pack_state<<<cdiv(count, 256), 256, 0, st>>>(R, first, count, out, changed_bit); }
}

}  // namespace b200vis

#ifdef B200VIS_TILE_TIMING
extern "C" __attribute__((visibility("default"))) int b200vis_debug_tile_timing(unsigned long long *out, unsigned n_ctas) {
    if (n_ctas > 8192u) n_ctas = 8192u;
    return (int)cudaMemcpyFromSymbol(out, b200vis::g_tile_timing, (size_t)n_ctas * 16 * sizeof(unsigned long long));
}
#endif
