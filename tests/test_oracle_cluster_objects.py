"""The CPU restatement of the clusterable-object spheres and of the per-kind ViewClusterBindings counters
(tests/cluster_objects_oracle.py): known answers, a float64 cross-check, and the counters against the list lengths."""
import math

import numpy as np

from bevy_b200 import scenes
import cluster_objects_oracle as coo
import oracle as orc


def _sphere(kind, gt, light_range=0.0):
    return coo.object_spheres([kind], gt, [light_range])[0]


def _gt(m3_columns, t=(1.0, 2.0, 3.0)):
    return np.concatenate([np.asarray(m3_columns, np.float32).reshape(-1), np.asarray(t, np.float32)])


def test_identity_probe_has_radius_sqrt3():
    for kind in (coo.REFLECTION_PROBE, coo.IRRADIANCE_VOLUME):
        s = _sphere(kind, orc.IDENTITY_GT)
        assert s[3] == np.float32(math.sqrt(3.0)) and (s[:3] == 0).all()


def test_decal_radius_is_the_length_of_the_scale_whatever_the_sign_of_the_determinant():
    for sx in (2.0, -2.0):
        s = _sphere(coo.DECAL, _gt(np.diag([sx, 3.0, 6.0])))
        assert s[3] == np.float32(7.0) and tuple(s[:3]) == (1.0, 2.0, 3.0)


def test_rect_and_point_light_ranges_pass_through():
    for kind in (coo.POINT_LIGHT, coo.RECT_LIGHT):
        for r in (0.3, 12.5, 1e-30):
            s = _sphere(kind, _gt(np.diag([2.0, -3.0, 0.5]), (4.0, 5.0, 6.0)), r)
            assert s[3] == np.float32(r) and tuple(s[:3]) == (4.0, 5.0, 6.0)


def _ulps(a, b):
    return abs(int(np.float32(a).view(np.int32)) - int(np.float32(b).view(np.int32)))


def test_rotated_probe_matches_float64_within_one_ulp():
    for axis in "xyz":
        for deg in range(0, 360, 15):
            gt = scenes.quat_to_gt(scenes.quat_axis(axis, math.radians(deg)), (7.0, -8.0, 9.0))
            m = gt[:9].astype(np.float64).reshape(3, 3)                                   # rows = the columns X, Y, Z
            s = _sphere(coo.REFLECTION_PROBE, gt)
            assert _ulps(s[3], np.linalg.norm(m.sum(0))) <= 1, (axis, deg)                # |X + Y + Z|
            assert tuple(s[:3]) == (7.0, -8.0, 9.0)


def test_scaled_probe_and_decal_stay_near_float64():
    """With non-uniform scales (some negative) the float32 sums round more often: a few ulps, never more."""
    rng = np.random.default_rng(18)
    q = scenes.random_unit_quats(rng, 200)
    for i in range(200):
        gt = scenes.quat_to_gt(q[i], rng.uniform(-100, 100, 3))
        scale = rng.uniform(0.1, 5.0, 3) * np.where(rng.random(3) < 0.3, -1.0, 1.0)
        gt[:9] = (gt[:9].reshape(3, 3) * scale[:, None]).reshape(-1).astype(np.float32)   # column k scaled by scale[k]
        m = gt[:9].astype(np.float64).reshape(3, 3)
        probe = _sphere(coo.REFLECTION_PROBE, gt)[3]
        assert _ulps(probe, np.linalg.norm(m.sum(0))) <= 4, i
        decal = _sphere(coo.DECAL, gt)[3]
        assert _ulps(decal, math.sqrt(float((m * m).sum()))) <= 4, i                      # |(|X|, |Y|, |Z|)|


def test_spot_lights_have_no_sphere_here():
    try:
        _sphere(1, orc.IDENTITY_GT, 1.0)
    except ValueError:
        return
    raise AssertionError("kind 1 must be refused")


def _random_clusters(rng, n_clusters, kinds):
    """CSR lists with ascending ordinals per cluster (the push order)."""
    offsets, indices = [0], []
    for _ in range(n_clusters):
        k = int(rng.integers(0, 12))
        indices.extend(sorted(rng.choice(len(kinds), size=min(k, len(kinds)), replace=False).tolist()))
        offsets.append(len(indices))
    return np.array(offsets, np.uint32), np.array(indices, np.uint32)


def test_kind_aware_bindings_count_every_entry_once():
    rng = np.random.default_rng(3)
    kinds = np.concatenate([np.zeros(20), np.full(6, 2), rng.choice([3, 4], 10), np.full(8, 5)]).astype(np.uint8)
    offsets, indices = _random_clusters(rng, 300, kinds)
    gmap = rng.permutation(len(kinds)).astype(np.uint32)
    oc, il, no, ni = coo.cluster_bindings_by_kind(offsets, indices, kinds, gmap)
    assert no == 300 and ni == len(indices)
    assert (oc[:, 0] == offsets[:-1]).all() and (oc[:, 2] == 0).all() and (oc[:, 7] == 0).all()
    assert (oc[:, 1:7].sum(1) == np.diff(offsets)).all()
    for c in range(300):
        got = kinds[indices[offsets[c]:offsets[c + 1]]]
        assert [int(oc[c, 1]), int(oc[c, 3]), int(oc[c, 4]), int(oc[c, 5]), int(oc[c, 6])] == \
               [int((got == k).sum()) for k in (0, 2, 3, 4, 5)]
    assert (il == gmap[indices]).all()


def test_kind_aware_bindings_of_point_lights_equal_the_point_light_packing():
    rng = np.random.default_rng(4)
    kinds = np.zeros(40, np.uint8)
    offsets, indices = _random_clusters(rng, 500, kinds)
    a = orc.cluster_bindings(offsets, indices, None, storage=True)
    b = coo.cluster_bindings_by_kind(offsets, indices, kinds)
    assert all(np.array_equal(x, y) for x, y in zip(a[:2], b[:2])) and a[2:] == b[2:]
