"""Synthetic scenes for BASELINE.json's configs (SURVEY.md section 8d).

All generators are deterministic (numpy PCG64, seed 42 unless stated) and
produce plain numpy columns in the layout of include/b200vis.h.  They restate
the reference's scene *specs* (examples/stress_tests/*.rs, benches/.../propagate.rs);
there is no network for real assets, so everything is synthetic.
"""
import math
from dataclasses import dataclass, field

import numpy as np

NO_PARENT = 0xFFFFFFFF
F_INHERITED_VISIBLE, F_HAS_AABB, F_HAS_SPHERE, F_SPHERE_FROM_GT = 0x01, 0x02, 0x04, 0x40
CLASS_MESH, CLASS_LIGHT = 0x01, 0x02      # VisibilityClass bits: Mesh3d, ClusterVisibilityClass


@dataclass
class Camera:
    gt: np.ndarray                 # [12] GlobalTransform (x_axis, y_axis, z_axis, translation)
    fov: float = math.pi / 4       # PerspectiveProjection::default (projection.rs:419-426)
    aspect: float = 16.0 / 9.0
    near: float = 0.1
    far: float = 1000.0
    quat: np.ndarray = None        # [4] rotation, kept for animation


@dataclass
class Scene:
    name: str
    parent: np.ndarray             # [n] u32
    trs: np.ndarray                # [n,10] f32
    bounds: np.ndarray             # [n,6] f32
    flags: np.ndarray              # [n] u8
    class_mask: np.ndarray         # [n] u8
    entity_bits: np.ndarray        # [n] u64
    light_row: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint32))
    light_range: np.ndarray = field(default_factory=lambda: np.zeros(0, np.float32))
    cameras: list = field(default_factory=list)
    roots: np.ndarray = None       # rows of hierarchy roots (the per-frame movers)
    screen: tuple = (1920, 1080)
    layer_mask: np.ndarray = None  # [n] u64 RenderLayers first block (None => default layer)
    range_mask: np.ndarray = None  # [n] u32 VisibleEntityRanges bitmask (None => resource absent)
    light_layers: np.ndarray = None
    view_layers: list = None       # per camera u64
    view_flags: list = None        # per camera B200VIS_VIEW_*
    view_range_index: list = None  # per camera i8

    @property
    def n(self):
        return len(self.parent)


# ---- quaternion helpers (float64 maths, float32 storage: inputs, not parity-critical) --------
def quat_mul(a, b):
    ax, ay, az, aw = a[..., 0], a[..., 1], a[..., 2], a[..., 3]
    bx, by, bz, bw = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    return np.stack([aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw,
                     aw * bw - ax * bx - ay * by - az * bz], axis=-1)


def quat_axis(axis, angle):
    q = np.zeros(4); q["xyz".index(axis)] = math.sin(angle / 2); q[3] = math.cos(angle / 2)
    return q


def quat_to_gt(q, t):
    """Affine3A from rotation + translation, float64 -> float32 (scale 1)."""
    x, y, z, w = [float(v) for v in q]
    X = (1 - 2 * (y * y + z * z), 2 * (x * y + w * z), 2 * (x * z - w * y))
    Y = (2 * (x * y - w * z), 1 - 2 * (x * x + z * z), 2 * (y * z + w * x))
    Z = (2 * (x * z + w * y), 2 * (y * z - w * x), 1 - 2 * (x * x + y * y))
    return np.array([*X, *Y, *Z, *t], np.float32)


def random_unit_quats(rng, n):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return q


def look_at_quats(pos, target=(0.0, 0.0, 0.0), up=(0.0, 1.0, 0.0)):
    """Transform::looking_at: back = -(target-pos).normalize(); right = up x back; up' = back x right."""
    pos = np.asarray(pos, np.float64)
    back = pos - np.asarray(target, np.float64)
    back /= np.linalg.norm(back, axis=1, keepdims=True)
    right = np.cross(np.asarray(up, np.float64)[None], back)
    nr = np.linalg.norm(right, axis=1, keepdims=True)
    right = np.where(nr > 1e-9, right / np.maximum(nr, 1e-30), np.array([[1.0, 0.0, 0.0]]))
    upv = np.cross(back, right)
    m = np.stack([right, upv, back], axis=2)          # columns
    # matrix -> quaternion (Shepperd), vectorised on the largest diagonal
    n = len(pos)
    q = np.zeros((n, 4))
    tr = m[:, 0, 0] + m[:, 1, 1] + m[:, 2, 2]
    s = np.sqrt(np.maximum(tr + 1.0, 1e-12)) * 2
    qa = np.stack([(m[:, 2, 1] - m[:, 1, 2]) / s, (m[:, 0, 2] - m[:, 2, 0]) / s, (m[:, 1, 0] - m[:, 0, 1]) / s, 0.25 * s], 1)
    sx = np.sqrt(np.maximum(1.0 + m[:, 0, 0] - m[:, 1, 1] - m[:, 2, 2], 1e-12)) * 2
    qb = np.stack([0.25 * sx, (m[:, 0, 1] + m[:, 1, 0]) / sx, (m[:, 0, 2] + m[:, 2, 0]) / sx, (m[:, 2, 1] - m[:, 1, 2]) / sx], 1)
    sy = np.sqrt(np.maximum(1.0 + m[:, 1, 1] - m[:, 0, 0] - m[:, 2, 2], 1e-12)) * 2
    qc = np.stack([(m[:, 0, 1] + m[:, 1, 0]) / sy, 0.25 * sy, (m[:, 1, 2] + m[:, 2, 1]) / sy, (m[:, 0, 2] - m[:, 2, 0]) / sy], 1)
    sz = np.sqrt(np.maximum(1.0 + m[:, 2, 2] - m[:, 0, 0] - m[:, 1, 1], 1e-12)) * 2
    qd = np.stack([(m[:, 0, 2] + m[:, 2, 0]) / sz, (m[:, 1, 2] + m[:, 2, 1]) / sz, 0.25 * sz, (m[:, 1, 0] - m[:, 0, 1]) / sz], 1)
    big = np.argmax(np.stack([tr, m[:, 0, 0], m[:, 1, 1], m[:, 2, 2]], 1), 1)
    q = np.where((big == 0)[:, None], qa, np.where((big == 1)[:, None], qb, np.where((big == 2)[:, None], qc, qd)))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return q


def fibonacci_sphere(n, radius):
    """fibonacci_spiral_on_sphere + spherical_polar_to_cartesian (many_cubes.rs:574-588), f64."""
    i = np.arange(n, dtype=np.float64)
    golden = 0.5 * (1.0 + math.sqrt(5.0))
    eps = 0.36
    theta = 2.0 * math.pi * (i / golden)
    phi = np.arccos(1.0 - 2.0 * (i + eps) / (n - 1.0 + 2.0 * eps))
    return radius * np.stack([np.cos(theta) * np.sin(phi), np.sin(theta) * np.sin(phi), np.cos(phi)], 1)


def _camera(yaw=0.0):
    q = quat_axis("y", yaw)
    return Camera(gt=quat_to_gt(q, (0.0, 0.0, 0.0)), quat=q)


def four_cameras():
    """Cameras at the origin looking -Z, +X... i.e. yaw 0, 90, 180, 270 degrees (config #3)."""
    return [_camera(k * math.pi / 2) for k in range(4)]


def _entity_bits(n, start=0):
    # Entity::to_bits() = index | generation << 32 with generation 0: ascending rows
    return (np.arange(n, dtype=np.uint64) + np.uint64(start))


def _trs(t, q=None, s=None):
    n = len(t)
    out = np.zeros((n, 10), np.float32)
    out[:, 0:3] = t
    out[:, 3:7] = (0, 0, 0, 1) if q is None else q
    out[:, 7:10] = 1.0 if s is None else s
    return out


def _lights(rng, n_lights, radius=50.0, range_lo=0.3, range_hi=20.0):
    """Point lights on the radius-50 Fibonacci sphere (many_lights.rs:48-86), log-uniform range."""
    pos = fibonacci_sphere(n_lights, radius).astype(np.float32)
    if range_hi > range_lo:
        rng_ = np.exp(rng.uniform(math.log(range_lo), math.log(range_hi), n_lights)).astype(np.float32)
    else:
        rng_ = np.full(n_lights, range_lo, np.float32)
    return pos, rng_


def _append_lights(scene_cols, pos, lrange):
    parent, trs, bounds, flags, cls = scene_cols
    n0, L = len(parent), len(pos)
    parent = np.concatenate([parent, np.full(L, NO_PARENT, np.uint32)])
    trs = np.concatenate([trs, _trs(pos)])
    b = np.zeros((L, 6), np.float32); b[:, 3] = lrange           # Sphere { center: GT.translation, radius: range }
    bounds = np.concatenate([bounds, b])
    flags = np.concatenate([flags, np.full(L, F_INHERITED_VISIBLE | F_HAS_SPHERE | F_SPHERE_FROM_GT, np.uint8)])
    cls = np.concatenate([cls, np.full(L, CLASS_LIGHT, np.uint8)])
    light_row = (n0 + np.arange(L)).astype(np.uint32)
    return (parent, trs, bounds, flags, cls), light_row


def forest(n_trees=3922, levels=8, n_lights=256, seed=42, name=None):
    """Config #3/#5: complete binary trees in BFS order per tree; roots U[-500,500]^3; local T U[-2,2]^3,
    uniform random rotation, uniform scale U[0.5,1.5]; Aabb half extents U[0.25,0.75]^3; 4 cameras;
    lights on the radius-50 sphere with log-uniform range 0.3..20."""
    rng = np.random.default_rng(seed)
    per = (1 << levels) - 1
    n = n_trees * per
    local = np.arange(per, dtype=np.int64)
    lp = np.where(local == 0, -1, (local - 1) // 2)
    base = (np.arange(n_trees, dtype=np.int64) * per)[:, None]
    parent = np.where(lp[None, :] < 0, NO_PARENT, base + lp[None, :]).astype(np.uint32).reshape(-1)
    t = rng.uniform(-2.0, 2.0, (n, 3))
    roots = (np.arange(n_trees) * per)
    t[roots] = rng.uniform(-500.0, 500.0, (n_trees, 3))
    q = random_unit_quats(rng, n)
    s = rng.uniform(0.5, 1.5, (n, 1)).repeat(3, 1)
    trs = _trs(t.astype(np.float32), q.astype(np.float32), s.astype(np.float32))
    bounds = np.zeros((n, 6), np.float32)
    bounds[:, 3:6] = rng.uniform(0.25, 0.75, (n, 3))
    flags = np.full(n, F_INHERITED_VISIBLE | F_HAS_AABB, np.uint8)
    cls = np.full(n, CLASS_MESH, np.uint8)
    cols = (parent, trs, bounds, flags, cls)
    light_row = np.zeros(0, np.uint32); lrange = np.zeros(0, np.float32)
    if n_lights:
        pos, lrange = _lights(rng, n_lights)
        cols, light_row = _append_lights(cols, pos, lrange)
    parent, trs, bounds, flags, cls = cols
    return Scene(name or f"forest_{n_trees}x{per}_L{n_lights}", parent, trs, bounds, flags, cls,
                 _entity_bits(len(parent)), light_row, lrange, four_cameras(), roots.astype(np.uint32))


def many_cubes(n=160_000, n_lights=0, light_range=(0.3, 0.3), seed=42, name=None):
    """Config #2 (and #4 with lights): Fibonacci sphere radius 500, each looking at the origin, flat;
    Aabb half extents r in [0.25, 0.75] per mesh kind (many_cubes.rs:187-206, 444-453); one camera."""
    rng = np.random.default_rng(seed)
    pos = fibonacci_sphere(n, 500.0)
    q = look_at_quats(pos)
    trs = _trs(pos.astype(np.float32), q.astype(np.float32))
    kinds = rng.uniform(0.25, 0.75, 16).astype(np.float32)        # a handful of mesh sizes, chosen per entity
    r = kinds[rng.integers(0, 16, n)]
    bounds = np.zeros((n, 6), np.float32); bounds[:, 3:6] = r[:, None]
    parent = np.full(n, NO_PARENT, np.uint32)
    flags = np.full(n, F_INHERITED_VISIBLE | F_HAS_AABB, np.uint8)
    cls = np.full(n, CLASS_MESH, np.uint8)
    cols = (parent, trs, bounds, flags, cls)
    light_row = np.zeros(0, np.uint32); lrange = np.zeros(0, np.float32)
    if n_lights:
        lpos, lrange = _lights(rng, n_lights, 50.0, light_range[0], light_range[1])
        cols, light_row = _append_lights(cols, lpos, lrange)
    parent, trs, bounds, flags, cls = cols
    return Scene(name or f"many_cubes_{n}_L{n_lights}", parent, trs, bounds, flags, cls, _entity_bits(len(parent)),
                 light_row, lrange, [_camera(0.0)], np.arange(0, n, max(n // 4096, 1), dtype=np.uint32))


def propagate_bench_scene():
    """Config #1: benches/benches/bevy_transform/propagate.rs:23-25, 74-82, 136-189: 48 roots x fan-out
    [4,4,3,3,2,2] (1077 nodes per tree, spawn order = BFS per tree) + 12000 flat entities."""
    fanout = [4, 4, 3, 3, 2, 2]
    parent, t = [], []
    roots = []
    for root_idx in range(48):
        r = len(parent); roots.append(r)
        parent.append(NO_PARENT); t.append((root_idx * 3.0, 0.0, 0.0))
        current = [r]
        for depth, fo in enumerate(fanout):
            nxt = []
            for p in current:
                for child_idx in range(fo):
                    seed = np.float32(root_idx * 7919 + depth * 313 + child_idx)
                    angle = np.float32(np.float32(seed * np.float32(0.11)) % np.float32(2 * math.pi))
                    c = len(parent)
                    parent.append(p)
                    t.append((math.cos(angle) * (depth + 1.0), math.sin(angle) * (depth + 0.5), depth * 0.75))
                    nxt.append(c)
            current = nxt
    for i in range(12000):
        parent.append(NO_PARENT); t.append((i * 0.001, 0.0, 0.0))
    n = len(parent)
    parent = np.array(parent, np.uint32)
    trs = _trs(np.array(t, np.float32))
    bounds = np.zeros((n, 6), np.float32); bounds[:, 3:6] = 0.5
    flags = np.full(n, F_INHERITED_VISIBLE | F_HAS_AABB, np.uint8)
    return Scene("propagate_bench_63696", parent, trs, bounds, flags, np.full(n, CLASS_MESH, np.uint8), _entity_bits(n),
                 cameras=[_camera(0.0)], roots=np.array(roots, np.uint32))


RECT_LIGHT, REFLECTION_PROBE, IRRADIANCE_VOLUME, DECAL = 2, 3, 4, 5   # ClusterableObjectType::ordering().0


def add_clusterable_objects(scene, n_rect=64, n_probe=128, n_decal=256, seed=7, hidden_frac=0.1,
                            rect_layer_choices=(1, 2, 3)):
    """Appends rect lights, light probes (reflection probes and irradiance volumes interleaved) and clustered decals to
    `scene`, in the reference's push order (assign.rs:231-295), and records them as scene.obj_kind / obj_row / obj_range /
    obj_layers.  Each object is a child of a random hierarchy root, so its GlobalTransform changes whenever the roots move,
    with a random rotation and a non-uniform scale whose x is negated for every third object (negative determinant).  All
    carry the unit-cube Aabb of add_light_probe_and_decal_aabbs (bevy_light/src/cluster/mod.rs:520-537), so the cull decides
    their ViewVisibility; `hidden_frac` of them are not InheritedVisibility-visible.  Rect lights get a log-uniform range and
    a RenderLayers mask drawn from `rect_layer_choices` (also their row's layer mask); probes and decals the default layer.
    The scene's columns are replaced by longer ones; the scene is returned."""
    rng = np.random.default_rng(seed)
    n_obj = n_rect + n_probe + n_decal
    kind = np.concatenate([np.full(n_rect, RECT_LIGHT), rng.choice([REFLECTION_PROBE, IRRADIANCE_VOLUME], n_probe),
                           np.full(n_decal, DECAL)]).astype(np.uint32)
    n0 = scene.n
    roots = scene.roots if scene.roots is not None and len(scene.roots) else np.zeros(0, np.uint32)
    parent = roots[rng.integers(0, len(roots), n_obj)].astype(np.uint32) if len(roots) else np.full(n_obj, NO_PARENT, np.uint32)
    s = rng.uniform(0.5, 3.0, (n_obj, 3))
    s[::3, 0] *= -1.0
    trs = _trs(rng.uniform(-3.0, 3.0, (n_obj, 3)).astype(np.float32), random_unit_quats(rng, n_obj).astype(np.float32),
               s.astype(np.float32))
    bounds = np.zeros((n_obj, 6), np.float32); bounds[:, 3:6] = 0.5
    flags = np.full(n_obj, F_INHERITED_VISIBLE | F_HAS_AABB, np.uint8)
    flags[rng.random(n_obj) < hidden_frac] = F_HAS_AABB
    obj_range = np.zeros(n_obj, np.float32)
    obj_range[:n_rect] = np.exp(rng.uniform(math.log(0.5), math.log(15.0), n_rect))
    obj_layers = np.ones(n_obj, np.uint64)
    obj_layers[:n_rect] = np.asarray(rect_layer_choices, np.uint64)[rng.integers(0, len(rect_layer_choices), n_rect)]
    layer_mask = np.ones(n0, np.uint64) if scene.layer_mask is None else scene.layer_mask
    scene.parent = np.concatenate([scene.parent, parent])
    scene.trs = np.concatenate([scene.trs, trs])
    scene.bounds = np.concatenate([scene.bounds, bounds])
    scene.flags = np.concatenate([scene.flags, flags])
    scene.class_mask = np.concatenate([scene.class_mask, np.full(n_obj, CLASS_LIGHT, np.uint8)])
    scene.entity_bits = np.concatenate([scene.entity_bits, _entity_bits(n_obj, int(scene.entity_bits.max()) + 1 if n0 else 0)])
    scene.layer_mask = np.concatenate([layer_mask, obj_layers])
    if scene.range_mask is not None:
        scene.range_mask = np.concatenate([scene.range_mask, np.zeros(n_obj, np.uint32)])
    scene.obj_kind, scene.obj_row = kind, (n0 + np.arange(n_obj)).astype(np.uint32)
    scene.obj_range, scene.obj_layers = obj_range, obj_layers
    scene.name = f"{scene.name}_O{n_rect}r{n_probe}p{n_decal}d"
    return scene


# ---- per-frame animation ---------------------------------------------------------------------
def advance_cameras(scene, delta=0.15 / 60.0):
    """move_camera (many_cubes.rs:590-603): rotate_z(delta) then rotate_x(delta); Transform::rotate
    pre-multiplies."""
    for cam in scene.cameras:
        q = quat_mul(quat_axis("z", delta), cam.quat)
        q = quat_mul(quat_axis("x", delta), q)
        cam.quat = q / np.linalg.norm(q)
        cam.gt = quat_to_gt(cam.quat, cam.gt[9:12])


def mutate_roots(scene, frame):
    """mutate_roots (propagate.rs:115-128) applied to every root: z += sin(phase)*0.02, rotate_y(0.0015).
    Returns (rows, trs_rows) to upload."""
    rows = scene.roots
    trs = scene.trs[rows]
    phase = (frame + np.arange(len(rows))) * 0.001
    trs[:, 2] += (np.sin(phase) * 0.02).astype(np.float32)
    q = quat_mul(quat_axis("y", 0.0015)[None], trs[:, 3:7].astype(np.float64))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    trs[:, 3:7] = q.astype(np.float32)
    scene.trs[rows] = trs
    return rows, trs
