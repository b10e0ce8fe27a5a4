"""CPU restatement of what assign_objects_to_clusters gathers for rect lights, light probes and clustered decals, and of the
per-kind counters they add to ViewClusterBindings (TEST INFRASTRUCTURE).

The per-cluster walk of these kinds is the point-light walk (assign.rs:740-800), so a frame's oracle is the existing
oracle.assign_lights_to_clusters over the visible point lights followed by the visible objects in ordinal order, each
given as the sphere `object_spheres` returns.

Floating point: numpy binary32 arrays, one IEEE rounding per ufunc and no contraction, in glam's SSE2 operation order
(SURVEY Appendix A); `np.sqrt` is correctly rounded.  glam order unverified (DESIGN.md §5)."""
import numpy as np

import oracle as orc

POINT_LIGHT, SPOT_LIGHT, RECT_LIGHT, REFLECTION_PROBE, IRRADIANCE_VOLUME, DECAL = 0, 1, 2, 3, 4, 5   # ordering().0 (assign.rs:115-131)


def _length(x, y, z):
    """Vec3A::length / Vec3::length: sqrt((x*x + y*y) + z*z)."""
    return np.sqrt((x * x + y * y) + z * z)


def object_spheres(kinds, gt, light_range=None):
    """(x, y, z, radius) per object, float32 [n, 4].
      kinds        ordering().0 per object: 0 point light (assign.rs:193-210), 2 rect light (:233-247), 3 reflection probe /
                   4 irradiance volume (:256-276), 5 decal (:279-295); spot lights (1) are not restated
      gt           [n, 12] GlobalTransforms (x_axis, y_axis, z_axis, translation); the centre is the translation for every kind
      light_range  PointLight::range / RectLight::range per object (read for kinds 0 and 2)
    Probe radius: transform.radius_vec3a(Vec3A::ONE) = (matrix3 * ONE).length() (global_transform.rs:252-254), with
    Mat3A * Vec3A = ((X*1) + (Y*1)) + (Z*1) lane-wise.  Decal radius: transform.scale().length() (:240-248) =
    Vec3(|X| * copysign(1, det), |Y|, |Z|).length(), det = Z . (X x Y) (glam Mat3A::determinant)."""
    kinds = np.asarray(kinds, np.uint32).reshape(-1)
    if (kinds == SPOT_LIGHT).any() or (kinds > DECAL).any():
        raise ValueError("object_spheres restates kinds 0, 2, 3, 4, 5 only")
    g = np.ascontiguousarray(gt, np.float32).reshape(-1, 12)
    X, Y, Z, T = g[:, 0:3], g[:, 3:6], g[:, 6:9], g[:, 9:12]
    one = np.float32(1.0)
    with np.errstate(over="ignore", invalid="ignore"):
        return _spheres(kinds, X, Y, Z, T, one, light_range)


def _spheres(kinds, X, Y, Z, T, one, light_range):
    v = (X * one + Y * one) + Z * one
    probe = _length(v[:, 0], v[:, 1], v[:, 2])
    # glam Vec3A::cross(X, Y) = (x.y*y.z - y.y*x.z, x.z*y.x - y.z*x.x, x.x*y.y - y.x*x.y), dotted with Z
    cross = np.stack([X[:, 1] * Y[:, 2] - Y[:, 1] * X[:, 2], X[:, 2] * Y[:, 0] - Y[:, 2] * X[:, 0],
                      X[:, 0] * Y[:, 1] - Y[:, 0] * X[:, 1]], 1)
    det = (Z[:, 0] * cross[:, 0] + Z[:, 1] * cross[:, 1]) + Z[:, 2] * cross[:, 2]
    sx = _length(X[:, 0], X[:, 1], X[:, 2]) * np.copysign(one, det)
    decal = _length(sx, _length(Y[:, 0], Y[:, 1], Y[:, 2]), _length(Z[:, 0], Z[:, 1], Z[:, 2]))
    rng = np.zeros(len(kinds), np.float32) if light_range is None else np.asarray(light_range, np.float32).reshape(-1)
    radius = np.where((kinds == POINT_LIGHT) | (kinds == RECT_LIGHT), rng,
                      np.where(kinds == DECAL, decal, probe)).astype(np.float32)
    return np.concatenate([T, radius[:, None]], 1).astype(np.float32)


def cluster_bindings_by_kind(offsets, indices, kinds, gpu_index_of_light=None):
    """STORAGE-mode ViewClusterBindings with ObjectsInClusterCpu's per-kind counters (bevy_light/src/cluster/mod.rs:478-512)
    in each header: (offset, point, spot, rect | probes, volumes, decals, 0) (bevy_pbr/src/cluster/mod.rs:636-652).
    kinds: ordering().0 per cluster ordinal.  The offsets and index list are oracle.cluster_bindings' own."""
    offsets = np.ascontiguousarray(offsets, np.uint32)
    indices = np.ascontiguousarray(indices, np.uint32)
    kinds = np.asarray(kinds, np.uint8)
    oc, il, no, ni = orc.cluster_bindings(offsets, indices, gpu_index_of_light, storage=True)
    oc = oc.copy()
    n = len(offsets) - 1
    cluster_of = np.repeat(np.arange(n), np.diff(offsets).astype(np.int64))
    counts = np.zeros((n, 6), np.uint32)
    np.add.at(counts, (cluster_of, kinds[indices].astype(np.int64)), 1)
    oc[:, 1:7] = counts
    return oc, il, no, ni
