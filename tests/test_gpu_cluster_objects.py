"""Rect lights, light probes and clustered decals in the cluster stage (b200vis_set_clusterable_objects), bit-exact against
the CPU oracle: cluster offsets and index lists, cluster_index_count, farthest_z bits, and -- through tests/parity.py's
compare_frame -- GlobalTransform, ViewVisibility and the visible lists, over several animated frames with the
MaxClusterableObjectRange feedback closed.  The oracle's input for a frame is the visible point lights, then the visible
objects in ordinal order, each as the sphere tests/cluster_objects_oracle.py restates (assign.rs:193-295).

The execution-mode switches (B200VIS_PIPELINE, B200VIS_CLUSTER_KERNEL) are read once per process, so each parity case runs
in its own interpreter."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import bevy_b200 as bb
from bevy_b200 import abi, scenes
import cluster_objects_oracle as coo
import oracle as orc
import parity

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


class ObjectsPipeline(bb.VisibilityPipeline):
    """VisibilityPipeline with the scene's clusterable objects set; clusters run whenever there are ordinals, also
    without point lights."""

    def __init__(self, scene, max_lights=None, **kw):
        n_ord = len(scene.light_row) + len(scene.obj_kind)
        super().__init__(scene, max_lights=max(n_ord, 1) if max_lights is None else max_lights, **kw)
        self.set_objects()

    def set_objects(self):
        sc = self.scene
        self.ctx.set_clusterable_objects(sc.obj_kind, sc.obj_row, sc.obj_range, sc.obj_layers)

    def clustered(self):
        return len(self.scene.light_row) + len(getattr(self.scene, "obj_kind", ())) > 0

    def update_views(self, clusters=True):
        views = []
        for v, cam in enumerate(self.scene.cameras):
            cfv = abi.host_perspective(cam.fov, cam.aspect, cam.near)
            frustum = abi.host_compute_frustum(cfv, cam.gt, cam.far)
            layers = 1 if self.scene.view_layers is None else int(self.scene.view_layers[v])
            views.append(abi.View.make(frustum, layers))
            if clusters and self.clustered():
                cv, scratch = abi.host_cluster_view_setup(self.cluster_config, cam.gt, cfv, frustum, layers, self.feedback[v])
                self._scratch[v], self.cluster_views[v] = scratch, cv
                self.ctx.set_cluster_view(v, cv)
        self.ctx.set_views(views)
        self.views = views

    def run_frame(self):
        self.ctx.run(abi.STAGE_ALL)


class ObjectsWorld(parity.OracleWorld):
    """The oracle side: parity.OracleWorld's propagate + cull, then assign_objects_to_clusters over the visible point lights
    followed by the visible objects."""

    def frame(self, views_planes, view_flags=None, cluster=True, mt=False):
        gt_changed, vv_changed, lists, _ = super().frame(views_planes, view_flags, cluster=False, mt=mt)
        sc = self.scene
        nl = len(sc.light_row)
        # the gathered order (assign.rs:193-295): point lights, then the objects; view_visibility.get() filters both
        rows = np.concatenate([np.asarray(sc.light_row, np.uint32), np.asarray(sc.obj_row, np.uint32)])
        kinds = self.kinds()
        rng = np.concatenate([np.asarray(sc.light_range, np.float32), np.asarray(sc.obj_range, np.float32)])
        light_layers = np.ones(nl, np.uint64) if sc.light_layers is None else np.asarray(sc.light_layers, np.uint64)
        all_layers = np.concatenate([light_layers, np.asarray(sc.obj_layers, np.uint64)])
        ords = np.nonzero(self.vv[rows] & 1)[0].astype(np.uint32)
        spheres = coo.object_spheres(kinds[ords], self.gt[rows[ords]], rng[ords])
        layers = np.ascontiguousarray(all_layers[ords], np.uint64)
        self.obj_clusters = []
        for v, cam in enumerate(sc.cameras):
            cfv = orc.perspective(cam.fov, cam.aspect, cam.near)
            vin = orc.default_cluster_view_in(cam.gt, cfv, views_planes[v], screen=sc.screen,
                                              view_layers=1 if sc.view_layers is None else int(sc.view_layers[v]),
                                              last_farthest_z=self.fb[v]["far"], last_index_count=self.fb[v]["cnt"],
                                              **self.cluster_kwargs)
            out, offsets, idx, _ = orc.assign_lights_to_clusters(vin, spheres, layers)
            self.fb[v]["far"] = out.farthest_z; self.fb[v]["cnt"] = out.total_index_count
            self.obj_clusters.append((out, offsets, ords[idx]))
        return gt_changed, vv_changed, lists, []

    def kinds(self):
        """ClusterableObjectType::ordering().0 of every cluster ordinal."""
        return np.concatenate([np.zeros(len(self.scene.light_row), np.uint8), np.asarray(self.scene.obj_kind, np.uint8)])


def check_clusters(tag, world, stats, get_clusters, dims):
    """get_clusters(v) -> (offsets, indices) of the device; dims(v) -> the device's grid."""
    for v, (out, offsets, idx) in enumerate(world.obj_clusters):
        assert tuple(dims(v)) == tuple(out.dims), f"{tag} view {v}: cluster dims {tuple(dims(v))} vs {tuple(out.dims)}"
        nc = out.dims[0] * out.dims[1] * out.dims[2]
        goff, gidx = get_clusters(v)
        assert (goff[:nc + 1] == offsets).all(), f"{tag} view {v}: cluster offsets differ"
        assert len(gidx) == len(idx) and (gidx == idx).all(), f"{tag} view {v}: cluster index lists differ ({len(gidx)} vs {len(idx)})"
        assert stats.cluster_index_count[v] == out.total_index_count, f"{tag} view {v}: index count"
        assert np.float32(stats.cluster_farthest_z[v]).view(np.uint32) == np.float32(out.farthest_z).view(np.uint32), \
            f"{tag} view {v}: farthest_z {stats.cluster_farthest_z[v]} vs {out.farthest_z}"


def compare_objects_frame(pipe, world, f):
    stats = parity.compare_frame(pipe, world, f, cluster=False)
    check_clusters(f"[{pipe.scene.name} frame {f}]", world, stats, pipe.ctx.download_clusters, lambda v: pipe.cluster_views[v].dims)
    return stats


def run_objects(scene, frames=4, before_frame=None, bindings=False, **kw):
    """Animated frames (roots move, cameras turn) compared with the oracle; returns the number of object entries seen."""
    pipe = ObjectsPipeline(scene, **kw)
    world = ObjectsWorld(scene)
    seen = 0
    try:
        if bindings:
            pipe.ctx.set_cluster_bindings(abi.BINDINGS_STORAGE, None)
        for f in range(frames):
            if f:
                scenes.advance_cameras(scene, 0.05)
                rows, trs = scenes.mutate_roots(scene, f)
                pipe.ctx.upload_transforms_scattered(rows, trs)
                world.tchanged[rows] = 1
            if before_frame is not None:
                before_frame(f, pipe, world)
            pipe.update_views()
            compare_objects_frame(pipe, world, f)
            nl = len(scene.light_row)
            for _, _, idx in world.obj_clusters:
                seen += int((idx >= nl).sum())
            if bindings:
                kinds = world.kinds()
                for v, (out, offsets, idx) in enumerate(world.obj_clusters):
                    w_oc, w_il, w_no, w_ni = coo.cluster_bindings_by_kind(offsets, idx, kinds)
                    g_oc, g_il, g_no, g_ni = pipe.ctx.download_cluster_bindings(v)
                    assert (g_no, g_ni) == (w_no, w_ni)
                    assert np.array_equal(g_oc, w_oc), f"frame {f} view {v}: offsets_and_counts differ"
                    assert np.array_equal(g_il, w_il), f"frame {f} view {v}: index lists differ"
                    assert (w_oc[:, 1:7].sum(1) == np.diff(offsets)).all()
    finally:
        pipe.close()
    return seen


def objects_scene(n_trees=300, n_lights=64, n_rect=64, n_probe=128, n_decal=256, seed=42):
    sc = scenes.forest(n_trees=n_trees, levels=8, n_lights=n_lights, seed=seed)
    scenes.add_clusterable_objects(sc, n_rect, n_probe, n_decal, seed=seed + 1)
    sc.view_layers = [1, 1, 3, 1]     # view 2 also renders layer 1: rect lights on layer 1 only are seen (and clustered) there
    return sc


# ---- the parity cases, one interpreter each --------------------------------------------------------------------------
def case_four_views():
    sc = objects_scene()
    kinds = set(sc.obj_kind.tolist())
    assert kinds == {2, 3, 4, 5} and (sc.flags[sc.obj_row] & bb.F_INHERITED_VISIBLE == 0).any()
    assert run_objects(sc, frames=4) > 0


def case_over_6400_ordinals():
    # 256 + 6600 ordinals: the fused kernel's distributed bit matrix holds at most 6400, so the split kernels run
    sc = objects_scene(n_trees=200, n_lights=256, n_rect=600, n_probe=3000, n_decal=3000, seed=11)
    assert run_objects(sc, frames=4) > 0


def case_changing_lists():
    sc = objects_scene(n_trees=200, n_lights=48, seed=5)
    full = (sc.obj_kind.copy(), sc.obj_row.copy(), sc.obj_range.copy(), sc.obj_layers.copy())
    lights = (sc.light_row.copy(), sc.light_range.copy())

    def before(f, pipe, world):
        if f == 2:       # probes gone: the decals move down to the rect lights
            keep = sc.obj_kind != 3
            sc.obj_kind, sc.obj_row, sc.obj_range, sc.obj_layers = (a[keep] for a in full)
            pipe.set_objects()
        if f == 3:       # half the point lights: every object ordinal shifts
            sc.light_row, sc.light_range = lights[0][::2], lights[1][::2]
            pipe.ctx.set_lights(sc.light_row, sc.light_range, None)
        if f == 4:       # everything back
            sc.obj_kind, sc.obj_row, sc.obj_range, sc.obj_layers = full
            pipe.set_objects()
            sc.light_row, sc.light_range = lights
            pipe.ctx.set_lights(sc.light_row, sc.light_range, None)
    assert run_objects(sc, frames=6, before_frame=before) > 0


def case_no_point_lights_run():
    sc = objects_scene(n_trees=250, n_lights=0, seed=9)
    assert run_objects(sc, frames=4) > 0


def case_no_point_lights_step():
    """b200vis_step with a result sink: the cluster stage runs on the objects alone, and the library's own feedback matches."""
    import torch
    sc = objects_scene(n_trees=250, n_lights=0, seed=13)
    pipe = ObjectsPipeline(sc)
    world = ObjectsWorld(sc)
    V = len(sc.cameras)
    cap = 1 << 20
    off = torch.zeros((V, 4097), dtype=torch.int32).pin_memory().numpy().view(np.uint32)
    idx = torch.zeros((V, cap), dtype=torch.int32).pin_memory().numpy().view(np.uint32)
    st_t = torch.zeros(ctypes.sizeof(bb.FrameStats), dtype=torch.uint8).pin_memory()
    st = bb.FrameStats.from_address(st_t.data_ptr())
    seen = 0
    try:
        pipe.ctx.set_result_sink(st_t.data_ptr(), None, off, idx)
        for f in range(5):
            rows = np.zeros(0, np.uint32); trs = np.zeros((0, 10), np.float32)
            if f:
                scenes.advance_cameras(sc, 0.05)
                rows, trs = scenes.mutate_roots(sc, f)
                rows = np.ascontiguousarray(rows, np.uint32); trs = np.ascontiguousarray(trs, np.float32)
                world.tchanged[rows] = 1
            arr = (bb.CameraDesc * V)()
            planes = []
            for v, cam in enumerate(sc.cameras):
                arr[v].global_transform[:] = cam.gt.tolist()
                arr[v].fov_y, arr[v].aspect, arr[v].near_z, arr[v].far_z = cam.fov, cam.aspect, cam.near, cam.far
                arr[v].layer_mask, arr[v].flags, arr[v].range_view_index = int(sc.view_layers[v]), bb.VIEW_ACTIVE, -1
                planes.append(abi.host_compute_frustum(abi.host_perspective(cam.fov, cam.aspect, cam.near), cam.gt, cam.far))
            _, _, lists, _ = world.frame(np.stack(planes))
            pipe.ctx.step(len(rows), rows.ctypes.data if len(rows) else 0, trs.ctypes.data if len(rows) else 0, arr, V,
                          pipe.cluster_config, wait=True)
            gt, _ = pipe.ctx.download_global_transforms(0, sc.n)
            assert (gt.view(np.uint32) == world.gt.view(np.uint32)).all(), f"frame {f}: GlobalTransform bits"
            vv, _ = pipe.ctx.download_view_visibility(0, sc.n)
            assert (vv == world.vv).all(), f"frame {f}: ViewVisibility"
            dims = [(ctypes.c_uint32 * 3)() for _ in range(V)]
            for v in range(V):
                assert pipe.ctx._lib.b200vis_cluster_view_dims(pipe.ctx._h, v, dims[v]) == 0
                assert (pipe.ctx.download_visible(v) == lists[v]).all()

            def sink_clusters(v):                  # the frame's CSR as the GPU wrote it into the pinned sink
                nc = dims[v][0] * dims[v][1] * dims[v][2]
                return off[v, :nc + 1], idx[v, :off[v, nc]]
            check_clusters(f"[step frame {f}]", world, st, sink_clusters, lambda v: tuple(dims[v]))
            seen += sum(len(c[2]) for c in world.obj_clusters)
        pipe.ctx.set_result_sink(None, None, None, None)
    finally:
        pipe.close()
    assert seen > 0


def case_storage_bindings():
    sc = objects_scene(n_trees=300, n_lights=64, seed=21)
    assert run_objects(sc, frames=4, bindings=True) > 0


VARIANTS = {
    "default": {},
    "serial": {"B200VIS_PIPELINE": "0"},
    "split": {"B200VIS_CLUSTER_KERNEL": "split"},
    "serial_split": {"B200VIS_PIPELINE": "0", "B200VIS_CLUSTER_KERNEL": "split"},
}


def run_case(name, env, timeout=600):
    e = dict(os.environ)
    for k in [k for k in e if k.startswith("B200VIS_")]:
        del e[k]
    e.update(env)
    prog = (f"import sys; sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {HERE!r})\n"
            f"import test_gpu_cluster_objects as t\nt.{name}()\n")
    res = subprocess.run([sys.executable, "-c", prog], env=e, capture_output=True, text=True, timeout=timeout)
    assert res.returncode == 0, f"{name} {env}\n{res.stdout[-2000:]}\n{res.stderr[-4000:]}"


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_objects_and_point_lights_on_four_views(variant):
    run_case("case_four_views", VARIANTS[variant])


@pytest.mark.parametrize("variant", ["default", "serial"])
def test_more_than_6400_ordinals_take_the_split_kernels(variant):
    run_case("case_over_6400_ordinals", VARIANTS[variant])


@pytest.mark.parametrize("variant", ["default", "serial", "split"])
def test_object_list_and_light_count_change_between_frames(variant):
    run_case("case_changing_lists", VARIANTS[variant])


@pytest.mark.parametrize("variant", ["default", "serial"])
def test_objects_without_point_lights_through_run(variant):
    run_case("case_no_point_lights_run", VARIANTS[variant])


@pytest.mark.parametrize("variant", ["default", "serial"])
def test_objects_without_point_lights_through_step_with_a_result_sink(variant):
    run_case("case_no_point_lights_step", VARIANTS[variant])


@pytest.mark.parametrize("variant", ["default", "split"])
def test_storage_bindings_count_each_kind(variant):
    run_case("case_storage_bindings", VARIANTS[variant])


# ---- refusals and teardown (in this interpreter) ----------------------------------------------------------------------
def _code(fn):
    try:
        fn()
    except bb.B200VisError as e:
        return e.code
    return 0


def test_error_paths():
    INVALID, CAPACITY, UNSUPPORTED = 1, 6, 8
    ctx = bb.Context(100, max_lights=8, max_views=1)
    try:
        ctx.set_lights([0, 1, 2], [1.0, 1.0, 1.0])
        ok = lambda k, r, g=None, l=None: _code(lambda: ctx.set_clusterable_objects(k, r, g, l))
        assert ok([2, 3, 4, 3, 5], [10, 11, 12, 13, 14], [1.0] * 5) == 0
        assert ok([2] * 6, list(range(10, 16)), [1.0] * 6) == CAPACITY          # 3 lights + 6 > 8
        assert _code(lambda: ctx.set_lights([0, 1, 2, 3], [1.0] * 4)) == CAPACITY   # 4 lights + the 5 objects set > 8
        assert ok([1], [10]) == UNSUPPORTED                                      # spot lights
        assert ok([0], [10]) == INVALID and ok([6], [10]) == INVALID
        assert ok([3, 2], [10, 11], [1.0, 1.0]) == INVALID                       # a rect light after a probe
        assert ok([5, 4], [10, 11]) == INVALID                                   # a probe after a decal
        assert ok([3, 4, 3], [10, 11, 12]) == 0                                  # probes and volumes interleave
        assert ok([5], [100]) == INVALID                                         # row >= max_entities
        assert ok([2], [10]) == INVALID                                          # a rect light without a range
        assert ok([3], [10]) == 0
        assert _code(lambda: ctx.set_cluster_bindings(abi.BINDINGS_UNIFORM)) == INVALID   # objects set: no uniform bindings
        assert ok([], []) == 0                                                   # n = 0 removes them
        ctx.set_cluster_bindings(abi.BINDINGS_UNIFORM)
        assert ok([3], [10]) == INVALID                                          # uniform bindings: no objects
        ctx.set_cluster_bindings(abi.BINDINGS_STORAGE)
        assert ok([3], [10]) == 0
        assert _code(lambda: ctx.set_lights([0, 1, 2, 3, 4, 5, 6], [1.0] * 7)) == 0   # 7 + 1 == 8 fits
    finally:
        ctx.close()
    multi = bb.Context(100, max_lights=8, max_views=1, world_size=2, rank=0)
    try:
        assert _code(lambda: multi.set_clusterable_objects([3], [10])) == UNSUPPORTED
        assert _code(lambda: multi.set_clusterable_objects([], [])) == 0
    finally:
        multi.close()


def test_removing_the_objects_equals_never_setting_them():
    """Objects set, two frames, then n = 0: every later frame's results and kernel-launch count equal those of a context that
    never had objects."""
    a_sc, b_sc = objects_scene(n_trees=120, n_lights=32, seed=3), objects_scene(n_trees=120, n_lights=32, seed=3)
    a = ObjectsPipeline(a_sc)
    b = bb.VisibilityPipeline(b_sc, max_lights=len(b_sc.light_row) + len(b_sc.obj_kind))
    try:
        deltas = {id(a): [], id(b): []}
        for f in range(7):
            if f == 2:
                a_sc.obj_kind, a_sc.obj_row = np.zeros(0, np.uint32), np.zeros(0, np.uint32)
                a.ctx.set_clusterable_objects([], [])
            for p in (a, b):
                if f:
                    scenes.advance_cameras(p.scene, 0.05)
                    rows, trs = scenes.mutate_roots(p.scene, f)
                    p.ctx.upload_transforms_scattered(rows, trs)
                p.update_views()
                p.ctx.synchronize()
                n0 = abi.kernel_launch_count()
                p.run_frame()
                p.ctx.synchronize()
                deltas[id(p)].append(abi.kernel_launch_count() - n0)
                p.read_feedback()
            if f < 3:
                continue
            sa, sb = a.ctx.download_frame_stats(), b.ctx.download_frame_stats()
            for v in range(len(a_sc.cameras)):
                assert sa.cluster_index_count[v] == sb.cluster_index_count[v] and sa.cluster_farthest_z[v] == sb.cluster_farthest_z[v]
                oa, ia = a.ctx.download_clusters(v); ob, ib = b.ctx.download_clusters(v)
                assert (oa == ob).all() and len(ia) == len(ib) and (ia == ib).all(), f"frame {f} view {v}"
                assert (a.ctx.download_visible(v) == b.ctx.download_visible(v)).all()
        assert deltas[id(a)][3:] == deltas[id(b)][3:], (deltas[id(a)], deltas[id(b)])
    finally:
        a.close(); b.close()
