"""ctypes binding of include/b200vis.h (one Python method per C entry point)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

NO_PARENT = 0xFFFFFFFF
DETACHED = 0xFFFFFFFE
F_INHERITED_VISIBLE, F_HAS_AABB, F_HAS_SPHERE, F_NO_FRUSTUM_CULLING = 0x01, 0x02, 0x04, 0x08
F_HAS_VIS_RANGE, F_NO_CPU_CULLING, F_SPHERE_FROM_GT = 0x10, 0x20, 0x40
VIEW_ACTIVE, VIEW_NO_CPU_CULLING = 0x01, 0x02
STAGE_PROPAGATE, STAGE_CULL, STAGE_CLUSTER_ASSIGN, STAGE_CLUSTER_LISTS = 0x1, 0x2, 0x4, 0x8
STAGE_CLUSTER = STAGE_CLUSTER_ASSIGN | STAGE_CLUSTER_LISTS
STAGE_ALL = 0xF
MAX_VIEWS = 8
MAX_CLUSTERS = 4096
# ClusterableObjectType::ordering().0 of the objects b200vis_set_clusterable_objects takes (assign.rs:115-131)
CLUSTERABLE_RECT_LIGHT, CLUSTERABLE_REFLECTION_PROBE, CLUSTERABLE_IRRADIANCE_VOLUME, CLUSTERABLE_DECAL = 2, 3, 4, 5
BINDINGS_OFF, BINDINGS_STORAGE, BINDINGS_UNIFORM = 0, 1, 2

ERR_NAMES = {1: "INVALID_ARG", 2: "CUDA", 3: "OUT_OF_MEMORY", 4: "HIERARCHY_CYCLE", 5: "PARENT_OUT_OF_RANGE",
             6: "CAPACITY", 7: "NOT_READY", 8: "UNSUPPORTED"}


class B200VisError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"b200vis error {code} ({ERR_NAMES.get(code, '?')}): {message}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_entities", C.c_uint32), ("max_lights", C.c_uint32),
                ("max_views", C.c_uint32), ("max_cluster_indices", C.c_uint32), ("world_size", C.c_uint32),
                ("rank", C.c_uint32), ("reserved", C.c_uint32)]


class View(C.Structure):
    _fields_ = [("half_spaces", (C.c_float * 4) * 6), ("layer_mask", C.c_uint64), ("flags", C.c_uint8),
                ("range_view_index", C.c_int8), ("pad", C.c_uint8 * 6)]

    @staticmethod
    def make(half_spaces, layer_mask=1, flags=VIEW_ACTIVE, range_view_index=-1):
        v = View()
        hs = np.ascontiguousarray(half_spaces, np.float32).reshape(6, 4)
        for i in range(6):
            for j in range(4):
                v.half_spaces[i][j] = hs[i, j]
        v.layer_mask = layer_mask; v.flags = flags; v.range_view_index = range_view_index
        return v


class ClusterView(C.Structure):
    _fields_ = [("enabled", C.c_uint32), ("dims", C.c_uint32 * 3), ("tile_size", C.c_uint32 * 2),
                ("is_orthographic", C.c_uint32), ("near_z", C.c_float), ("far_z", C.c_float),
                ("cluster_factors", C.c_float * 2), ("view_from_world", C.c_float * 16),
                ("clip_from_view", C.c_float * 16), ("view_from_world_scale", C.c_float * 3),
                ("view_from_world_scale_max", C.c_float), ("frustum", (C.c_float * 4) * 6),
                ("layer_mask", C.c_uint64), ("x_planes", C.POINTER(C.c_float)), ("y_planes", C.POINTER(C.c_float)),
                ("z_planes", C.POINTER(C.c_float))]


class ClusterConfig(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("dims", C.c_uint32 * 3), ("total", C.c_uint32), ("z_slices", C.c_uint32),
                ("first_slice_depth", C.c_float), ("far_z_mode", C.c_uint32), ("far_z_constant", C.c_float),
                ("dynamic_resizing", C.c_uint32), ("screen_w", C.c_uint32), ("screen_h", C.c_uint32),
                ("view_cluster_bindings_max_indices", C.c_uint32)]


class ClusterFeedback(C.Structure):
    _fields_ = [("has_farthest_z", C.c_uint32), ("farthest_z", C.c_float), ("has_index_count", C.c_uint32),
                ("index_count", C.c_uint32)]


class CameraDesc(C.Structure):
    _fields_ = [("global_transform", C.c_float * 12), ("fov_y", C.c_float), ("aspect", C.c_float), ("near_z", C.c_float),
                ("far_z", C.c_float), ("layer_mask", C.c_uint64), ("flags", C.c_uint8), ("range_view_index", C.c_int8),
                ("pad", C.c_uint8 * 6)]


class FrameStats(C.Structure):
    _fields_ = [("visible_count", C.c_uint32 * MAX_VIEWS), ("cluster_index_count", C.c_uint32 * MAX_VIEWS),
                ("cluster_farthest_z", C.c_float * MAX_VIEWS), ("cluster_index_overflow", C.c_uint32 * MAX_VIEWS),
                ("gt_changed_count", C.c_uint32), ("vv_changed_count", C.c_uint32), ("frame", C.c_uint32),
                ("pad", C.c_uint32)]


class ColumnSinks(C.Structure):
    _fields_ = [("global_transforms", C.c_void_p), ("gt_stride_floats", C.c_uint32), ("gt_changed_bits", C.c_void_p),
                ("view_visibility", C.c_void_p), ("vv_changed_bits", C.c_void_p)]


class ShadowItem(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("light_row", C.c_uint32), ("range", C.c_float), ("range_view_index", C.c_int32),
                ("layer_mask", C.c_uint64), ("frusta", C.c_float * 144)]


class ResultSink(C.Structure):
    _fields_ = [("stats", C.POINTER(FrameStats)), ("visible_rows", C.c_void_p), ("visible_capacity", C.c_uint32),
                ("visible_classes", C.c_void_p), ("cluster_offsets", C.c_void_p), ("cluster_indices", C.c_void_p), ("cluster_capacity", C.c_uint32)]


_lib = None
_P = C.POINTER
_vp = C.c_void_p

_SIGNATURES = {
    "b200vis_abi_version": (C.c_int32, []),
    "b200vis_struct_sizes": (None, [_P(C.c_uint32)]),
    "b200vis_create": (C.c_int32, [_P(Config), _P(_vp)]),
    "b200vis_destroy": (None, [_vp]),
    "b200vis_last_error": (C.c_char_p, [_vp]),
    "b200vis_set_stream": (C.c_int32, [_vp, _vp]),
    "b200vis_synchronize": (C.c_int32, [_vp]),
    "b200vis_join": (C.c_int32, [_vp]),
    "b200vis_tail_stream": (C.c_int32, [_vp, _P(_vp)]),
    "b200vis_set_topology": (C.c_int32, [_vp, C.c_uint32, _vp, _vp]),
    "b200vis_kernel_launch_count": (C.c_uint64, []),
    "b200vis_p2p_link": (C.c_int32, [_vp, C.c_uint32]),
    "b200vis_upload_render_layers_ext": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_set_view_render_layers_ext": (C.c_int32, [_vp, C.c_uint32, _vp]),
    "b200vis_set_shadow_items": (C.c_int32, [_vp, C.c_uint32, _vp, C.c_uint32]),
    "b200vis_download_visible_classes": (C.c_int32, [_vp, C.c_uint32, _vp, C.c_uint32, _P(C.c_uint32)]),
    "b200vis_cluster_view_dims": (C.c_int32, [_vp, C.c_uint32, _P(C.c_uint32)]),
    "b200vis_set_column_sinks": (C.c_int32, [_vp, _P(ColumnSinks)]),
    "b200vis_writeback_columns": (C.c_int32, [_vp]),
    "b200vis_writeback_columns_ex": (C.c_int32, [_vp, C.c_uint32]),
    "b200vis_host_plan_summary": (C.c_int32, [C.c_uint32, _vp, _P(C.c_uint32)]),
    "b200vis_host_tile_plan": (C.c_int32, [C.c_uint32, _vp, C.c_uint32, C.c_uint32, _P(C.c_uint32), _vp, _vp]),
    "b200vis_host_warp_plan": (C.c_int32, [C.c_uint32, _vp, C.c_uint32, C.c_uint32, _P(C.c_uint32), _vp, _vp, _vp, _vp]),
    "b200vis_plan_row_order": (C.c_int32, [C.c_uint32, _vp, _vp]),
    "b200vis_upload_transforms": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_upload_transforms_scattered": (C.c_int32, [_vp, C.c_uint32, _vp, _vp]),
    "b200vis_mark_transforms_changed": (C.c_int32, [_vp, C.c_uint32, C.c_uint32]),
    "b200vis_upload_global_transforms": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_upload_bounds": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp, _vp, _vp]),
    "b200vis_upload_view_visibility": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_set_static_transform_optimizations": (C.c_int32, [_vp, C.c_int32]),
    "b200vis_set_views": (C.c_int32, [_vp, C.c_uint32, _P(View)]),
    "b200vis_set_view_count": (C.c_int32, [_vp, C.c_uint32]),
    "b200vis_update_camera": (C.c_int32, [_vp, C.c_uint32, _P(CameraDesc), _P(ClusterConfig), _P(ClusterFeedback), _P(ClusterView)]),
    "b200vis_download_frame": (C.c_int32, [_vp, _P(FrameStats), _vp, C.c_uint32, _vp, _vp, C.c_uint32]),
    "b200vis_set_lights": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, _vp]),
    "b200vis_set_clusterable_objects": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, _vp, _vp]),
    "b200vis_set_cluster_view": (C.c_int32, [_vp, C.c_uint32, _P(ClusterView)]),
    "b200vis_record_frame_constants": (C.c_int32, [_vp, _P(C.c_uint32)]),
    "b200vis_use_recorded_frame_constants": (C.c_int32, [_vp, C.c_int32]),
    "b200vis_set_profiling": (C.c_int32, [_vp, C.c_int32]),
    "b200vis_collect_stage_times_ms": (C.c_int32, [_vp, _P(C.c_float), _P(C.c_float), _P(C.c_float), _P(C.c_uint32)]),
    "b200vis_step": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, C.c_uint32, _P(CameraDesc), _P(ClusterConfig), C.c_uint32]),
    "b200vis_run": (C.c_int32, [_vp, C.c_uint32]),
    "b200vis_download_frame_stats": (C.c_int32, [_vp, _P(FrameStats)]),
    "b200vis_download_global_transforms": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, C.c_uint32, _vp]),
    "b200vis_download_view_visibility": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "b200vis_download_visible": (C.c_int32, [_vp, C.c_uint32, _vp, C.c_uint32, _P(C.c_uint32)]),
    "b200vis_download_clusters": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, C.c_uint32, _P(C.c_uint32)]),
    "b200vis_set_result_sink": (C.c_int32, [_vp, _P(ResultSink)]),
    "b200vis_upload_shadow_casters": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_set_shadow_lights": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, _vp, C.c_int32, C.c_uint32]),
    "b200vis_run_shadow_culling": (C.c_int32, [_vp]),
    "b200vis_download_shadow_visible": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, C.c_uint32, _P(C.c_uint32)]),
    "b200vis_host_point_light_frusta": (None, [_vp, C.c_float, C.c_float, _vp]),
    "b200vis_upload_visibility_ranges": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "b200vis_set_visibility_range_views": (C.c_int32, [_vp, C.c_uint32, _vp]),
    "b200vis_download_visibility_ranges": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_upload_visibility": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_propagate_visibility": (C.c_int32, [_vp]),
    "b200vis_download_inherited_visibility": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "b200vis_set_cluster_bindings": (C.c_int32, [_vp, C.c_uint32, _vp, C.c_uint32]),
    "b200vis_download_cluster_bindings": (C.c_int32, [_vp, C.c_uint32, _vp, C.c_uint32, _vp, C.c_uint32, _P(C.c_uint32), _P(C.c_uint32)]),
    "b200vis_enable_visible_diff": (C.c_int32, [_vp, C.c_int32]),
    "b200vis_download_visible_diff": (C.c_int32, [_vp, C.c_uint32, _vp, C.c_uint32, _P(C.c_uint32), _vp, C.c_uint32, _P(C.c_uint32)]),
    "b200vis_set_visible_diff_sink": (C.c_int32, [_vp, _vp, C.c_uint32, _vp]),
    "b200vis_comm_unique_id": (C.c_int32, [_vp]),
    "b200vis_comm_init": (C.c_int32, [_vp, _vp]),
    "b200vis_p2p_export": (C.c_int32, [_vp, _vp]),
    "b200vis_p2p_import": (C.c_int32, [_vp, _vp]),
    "b200vis_cluster_exchange_bytes": (C.c_int32, [_vp, _P(C.c_size_t)]),
    "b200vis_set_cluster_exchange_buffers": (C.c_int32, [_vp, _vp, _vp]),
    "b200vis_host_perspective": (None, [C.c_float, C.c_float, C.c_float, _vp]),
    "b200vis_host_compute_frustum": (None, [_vp, _vp, C.c_float, _vp]),
    "b200vis_host_z_slice_thresholds": (None, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "b200vis_host_default_cluster_config": (None, [_P(ClusterConfig), C.c_uint32, C.c_uint32]),
    "b200vis_host_cluster_view_setup": (C.c_int32, [_P(ClusterConfig), _vp, _vp, _vp, C.c_uint64,
                                                    _P(ClusterFeedback), _vp, _P(ClusterView)]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def host_point_light_frusta(light_gt12, light_range, shadow_map_near_z=0.1):
    """update_point_light_frusta for one light -> [6, 6, 4] (no GPU needed)."""
    g = np.ascontiguousarray(light_gt12, np.float32)
    out = np.zeros((6, 6, 4), np.float32)
    load_library().b200vis_host_point_light_frusta(_ptr(g), float(light_range), float(shadow_map_near_z), _ptr(out))
    return out


def library_path():
    # B200VIS_LIB selects another build of the same ABI (kernel tuning experiments); the default is the in-tree library
    return os.environ.get("B200VIS_LIB") or os.path.join(_HERE, "libb200vis.so")


def load_library():
    """Loads the in-tree libb200vis.so.  Fails loudly if it has not been built."""
    global _lib
    if _lib is None:
        path = library_path()
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} is missing: run `python -m bevy_b200.build` (there is no CPU fallback)")
        lib = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def kernel_launch_count():
    return int(load_library().b200vis_kernel_launch_count())


def abi_version():
    return load_library().b200vis_abi_version()


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


def _arr(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def host_perspective(fov_y, aspect, near):
    out = np.zeros(16, np.float32)
    load_library().b200vis_host_perspective(fov_y, aspect, near, _ptr(out))
    return out


def host_compute_frustum(clip_from_view, camera_gt12, far):
    cfv = _arr(clip_from_view, np.float32); g = _arr(camera_gt12, np.float32); out = np.zeros((6, 4), np.float32)
    load_library().b200vis_host_compute_frustum(_ptr(cfv), _ptr(g), far, _ptr(out))
    return out


def host_z_slice_thresholds(factors, z_slices, ortho=False):
    f = _arr(factors, np.float32); out = np.zeros(max(z_slices - 1, 1), np.float32)
    load_library().b200vis_host_z_slice_thresholds(_ptr(f), z_slices, int(ortho), _ptr(out))
    return out[:max(z_slices - 1, 0)]


def host_default_cluster_config(w=1920, h=1080):
    cfg = ClusterConfig()
    load_library().b200vis_host_default_cluster_config(C.byref(cfg), w, h)
    return cfg


def host_cluster_view_setup(cfg, camera_gt12, clip_from_view, frustum, layer_mask=1, feedback=None):
    """Returns (ClusterView, scratch) -- keep `scratch` alive while the view is in use."""
    g = _arr(camera_gt12, np.float32); cfv = _arr(clip_from_view, np.float32); fr = _arr(frustum, np.float32)
    scratch = np.zeros(3 * 4097 * 4, np.float32)
    out = ClusterView()
    rc = load_library().b200vis_host_cluster_view_setup(C.byref(cfg), _ptr(g), _ptr(cfv), _ptr(fr), layer_mask,
                                                        None if feedback is None else C.byref(feedback),
                                                        _ptr(scratch), C.byref(out))
    if rc:
        raise B200VisError(rc, "b200vis_host_cluster_view_setup")
    return out, scratch


def host_plan_summary(parent):
    """(tiles, passes, max in-tile levels, rows with a parent in another tile) of the execution plan."""
    parent = _arr(parent, np.uint32); out = (C.c_uint32 * 4)()
    rc = load_library().b200vis_host_plan_summary(len(parent), _ptr(parent), out)
    if rc:
        raise B200VisError(rc, load_library().b200vis_last_error(None).decode())
    return tuple(out)


def host_tile_plan(parent, tile_rows=0):
    """The CTA-per-tile plan (b200vis_host_tile_plan): (tile_desc[T,8], topo[n]); desc columns = base, rows, levels,
    warp_sync_mask, top_levels, lvl_warps lo, lvl_warps hi, pass."""
    parent = _arr(parent, np.uint32)
    lib = load_library()
    nt = C.c_uint32(0)
    rc = lib.b200vis_host_tile_plan(len(parent), _ptr(parent), tile_rows, 0, C.byref(nt), None, None)
    if rc:
        raise B200VisError(rc, "host_tile_plan")
    T = nt.value
    desc = np.zeros((T, 8), np.uint32); topo = np.zeros(len(parent), np.uint32)
    rc = lib.b200vis_host_tile_plan(len(parent), _ptr(parent), tile_rows, T, C.byref(nt), _ptr(desc), _ptr(topo))
    if rc:
        raise B200VisError(rc, "host_tile_plan")
    return desc, topo


def host_warp_plan(parent, tile_rows=0):
    """The warp-per-tile plan (b200vis_host_warp_plan): (tile_desc[T,4], nonroot[T,8], sched[T,256], wtopo[n])."""
    parent = _arr(parent, np.uint32)
    lib = load_library()
    nt = C.c_uint32(0)
    rc = lib.b200vis_host_warp_plan(len(parent), _ptr(parent), tile_rows, 0, C.byref(nt), None, None, None, None)
    if rc:
        raise B200VisError(rc, "host_warp_plan")
    T = nt.value
    desc = np.zeros((T, 4), np.uint32); nonroot = np.zeros((T, 8), np.uint32)
    sched = np.zeros((T, 256), np.uint8); wtopo = np.zeros(len(parent), np.uint32)
    rc = lib.b200vis_host_warp_plan(len(parent), _ptr(parent), tile_rows, T, C.byref(nt), _ptr(desc), _ptr(nonroot), _ptr(sched), _ptr(wtopo))
    if rc:
        raise B200VisError(rc, "host_warp_plan")
    return desc, nonroot, sched, wtopo


def p2p_link(contexts):
    """b200vis_p2p_link: contexts[r] was created with world_size=len(contexts), rank=r (one process, several devices)."""
    arr = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
    rc = load_library().b200vis_p2p_link(arr, len(contexts))
    if rc:
        raise B200VisError(rc, contexts[0]._last_error() if hasattr(contexts[0], "_last_error") else "p2p_link")


def plan_row_order(parent):
    parent = _arr(parent, np.uint32); out = np.zeros(len(parent), np.uint32)
    rc = load_library().b200vis_plan_row_order(len(parent), _ptr(parent), _ptr(out))
    if rc:
        raise B200VisError(rc, "b200vis_plan_row_order")
    return out


class Context:
    """One b200vis_ctx.  Method names follow the C ABI one to one."""

    def __init__(self, max_entities, max_lights=0, max_views=1, device=0, max_cluster_indices=0, world_size=1, rank=0):
        self._lib = load_library()
        self._h = _vp()
        cfg = Config(device, max_entities, max_lights, max_views, max_cluster_indices, world_size, rank, 0)
        rc = self._lib.b200vis_create(C.byref(cfg), C.byref(self._h))
        if rc:
            raise B200VisError(rc, self._lib.b200vis_last_error(None).decode())
        self.max_entities, self.max_lights, self.max_views = max_entities, max_lights, max_views
        self._keep = []

    def close(self):
        if self._h:
            self._lib.b200vis_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise B200VisError(rc, self._lib.b200vis_last_error(self._h).decode())

    def set_stream(self, cuda_stream):
        self._check(self._lib.b200vis_set_stream(self._h, _vp(cuda_stream)))

    def tail_stream(self):
        s = _vp()
        self._check(self._lib.b200vis_tail_stream(self._h, C.byref(s)))
        return s.value or 0

    def join(self):
        self._check(self._lib.b200vis_join(self._h))

    def synchronize(self):
        self._check(self._lib.b200vis_synchronize(self._h))

    def set_topology(self, parent_row, entity_bits):
        p = _arr(parent_row, np.uint32); e = _arr(entity_bits, np.uint64)
        assert len(p) == len(e)
        self._check(self._lib.b200vis_set_topology(self._h, len(p), _ptr(p), _ptr(e)))
        self.n = len(p)

    def upload_transforms(self, first_row, trs):
        t = _arr(trs, np.float32).reshape(-1, 10)
        self._check(self._lib.b200vis_upload_transforms(self._h, first_row, len(t), _ptr(t)))

    def upload_transforms_raw(self, first_row, count, host_ptr):
        """trs at a raw host address (e.g. pinned memory): no numpy conversion on the hot path."""
        self._check(self._lib.b200vis_upload_transforms(self._h, first_row, count, _vp(host_ptr)))

    def upload_transforms_scattered(self, rows, trs):
        r = _arr(rows, np.uint32); t = _arr(trs, np.float32).reshape(-1, 10)
        assert len(r) == len(t)
        self._check(self._lib.b200vis_upload_transforms_scattered(self._h, len(r), _ptr(r), _ptr(t)))

    def upload_transforms_scattered_raw(self, count, rows_ptr, trs_ptr):
        self._check(self._lib.b200vis_upload_transforms_scattered(self._h, count, _vp(rows_ptr), _vp(trs_ptr)))

    def mark_transforms_changed(self, first_row, count):
        self._check(self._lib.b200vis_mark_transforms_changed(self._h, first_row, count))

    def upload_global_transforms(self, first_row, gt):
        g = _arr(gt, np.float32).reshape(-1, 12)
        self._check(self._lib.b200vis_upload_global_transforms(self._h, first_row, len(g), _ptr(g)))

    def upload_bounds(self, first_row, bounds, flags, class_mask, layer_mask=None, range_mask=None):
        b = _arr(bounds, np.float32).reshape(-1, 6); f = _arr(flags, np.uint8); c = _arr(class_mask, np.uint8)
        l = _arr(layer_mask, np.uint64); r = _arr(range_mask, np.uint32)
        self._check(self._lib.b200vis_upload_bounds(self._h, first_row, len(b), _ptr(b), _ptr(f), _ptr(c), _ptr(l), _ptr(r)))

    def upload_render_layers_ext(self, first_row, blocks):
        blocks = _arr(blocks, np.uint64).reshape(-1, 3)
        self._check(self._lib.b200vis_upload_render_layers_ext(self._h, first_row, len(blocks), _ptr(blocks)))

    def set_view_render_layers_ext(self, view, blocks):
        b = _arr(blocks, np.uint64).reshape(3)
        self._check(self._lib.b200vis_set_view_render_layers_ext(self._h, view, _ptr(b)))

    def upload_view_visibility(self, first_row, vv):
        v = _arr(vv, np.uint8)
        self._check(self._lib.b200vis_upload_view_visibility(self._h, first_row, len(v), _ptr(v)))

    def set_static_transform_optimizations(self, enabled):
        self._check(self._lib.b200vis_set_static_transform_optimizations(self._h, int(bool(enabled))))

    def set_views(self, views):
        arr = (View * max(len(views), 1))(*views)
        self._check(self._lib.b200vis_set_views(self._h, len(views), arr))
        self.n_views = len(views)

    def set_view_count(self, n):
        self._check(self._lib.b200vis_set_view_count(self._h, n))
        self.n_views = n

    def update_camera(self, view, camera_desc, cluster_config=None, feedback=None, out=None):
        self._check(self._lib.b200vis_update_camera(self._h, view, C.byref(camera_desc),
                                                    None if cluster_config is None else C.byref(cluster_config),
                                                    None if feedback is None else C.byref(feedback),
                                                    None if out is None else C.byref(out)))

    def download_frame(self, stats, visible_rows, cluster_offsets, cluster_indices):
        """One batched read-back into caller-owned (ideally pinned) numpy arrays:
        visible_rows [V, cap_v], cluster_offsets [V, 4097], cluster_indices [V, cap_c]."""
        self._check(self._lib.b200vis_download_frame(
            self._h, C.byref(stats), _ptr(visible_rows), 0 if visible_rows is None else visible_rows.shape[1],
            _ptr(cluster_offsets), _ptr(cluster_indices), 0 if cluster_indices is None else cluster_indices.shape[1]))

    def set_lights(self, light_row, light_range, layer_mask=None):
        r = _arr(light_row, np.uint32); g = _arr(light_range, np.float32); l = _arr(layer_mask, np.uint64)
        self._check(self._lib.b200vis_set_lights(self._h, len(r), _ptr(r), _ptr(g), _ptr(l)))

    def set_clusterable_objects(self, kind, row, rect_range=None, layer_mask=None):
        """Rect lights, light probes and clustered decals (kinds CLUSTERABLE_*), grouped in the reference's push order; object j
        becomes cluster ordinal n_lights + j.  rect_range / layer_mask: one entry per object, read for rect lights only.
        Empty arrays remove the objects."""
        k = _arr(kind, np.uint32); r = _arr(row, np.uint32)
        assert len(k) == len(r)
        g = _arr(rect_range, np.float32); l = _arr(layer_mask, np.uint64)
        assert g is None or len(g) == len(k)
        assert l is None or len(l) == len(k)
        self._check(self._lib.b200vis_set_clusterable_objects(self._h, len(k), _ptr(k), _ptr(r), _ptr(g), _ptr(l)))

    def cluster_dims(self, view):
        """Number of clusters of the view's current grid (0 = clustering off)."""
        d = (C.c_uint32 * 3)()
        self._check(self._lib.b200vis_cluster_view_dims(self._h, view, d))
        return int(d[0]) * int(d[1]) * int(d[2])

    def set_cluster_view(self, view, cluster_view):
        self._check(self._lib.b200vis_set_cluster_view(self._h, view, C.byref(cluster_view)))

    def record_frame_constants(self):
        slot = C.c_uint32(0)
        self._check(self._lib.b200vis_record_frame_constants(self._h, C.byref(slot)))
        return slot.value

    def use_recorded_frame_constants(self, slot):
        self._check(self._lib.b200vis_use_recorded_frame_constants(self._h, -1 if slot is None else int(slot)))

    def set_profiling(self, enabled):
        self._check(self._lib.b200vis_set_profiling(self._h, int(bool(enabled))))

    def collect_stage_times_ms(self):
        """(tile_ms, expand_ms, cluster_ms, frames): sums over the runs recorded since the last collect."""
        a, b_, c, n = C.c_float(0), C.c_float(0), C.c_float(0), C.c_uint32(0)
        self._check(self._lib.b200vis_collect_stage_times_ms(self._h, C.byref(a), C.byref(b_), C.byref(c), C.byref(n)))
        return a.value, b_.value, c.value, n.value

    def step(self, n_changed, rows_ptr, trs_ptr, cameras, n_cameras, cluster_config=None, wait=True, writeback=False):
        """b200vis_step: `cameras` is a ctypes array of CameraDesc."""
        self._check(self._lib.b200vis_step(self._h, n_changed, _vp(rows_ptr), _vp(trs_ptr), n_cameras, cameras,
                                           None if cluster_config is None else C.byref(cluster_config),
                                           (1 if wait else 0) | (2 if writeback else 0)))

    def run(self, stages=STAGE_ALL):
        self._check(self._lib.b200vis_run(self._h, stages))

    def download_frame_stats(self):
        s = FrameStats()
        self._check(self._lib.b200vis_download_frame_stats(self._h, C.byref(s)))
        return s

    def download_global_transforms(self, first_row, count, stride=12, want_changed=True):
        gt = np.zeros((count, stride), np.float32)
        ch = np.zeros(count, np.uint8) if want_changed else None
        self._check(self._lib.b200vis_download_global_transforms(self._h, first_row, count, _ptr(gt), stride, _ptr(ch)))
        return gt, ch

    def download_view_visibility(self, first_row, count):
        vv = np.zeros(count, np.uint8); ch = np.zeros(count, np.uint8)
        self._check(self._lib.b200vis_download_view_visibility(self._h, first_row, count, _ptr(vv), _ptr(ch)))
        return vv, ch

    def download_visible(self, view):
        cnt = C.c_uint32(0)
        self._check(self._lib.b200vis_download_visible(self._h, view, None, 0, C.byref(cnt)))
        rows = np.zeros(max(cnt.value, 1), np.uint32)
        self._check(self._lib.b200vis_download_visible(self._h, view, _ptr(rows), len(rows), C.byref(cnt)))
        return rows[:cnt.value]

    # ---- SURVEY 8(f) N3 ----
    def upload_shadow_casters(self, first, caster):
        c = np.ascontiguousarray(caster, np.uint8)
        self._check(self._lib.b200vis_upload_shadow_casters(self._h, first, len(c), _ptr(c)))

    def set_shadow_lights(self, light_ordinals, frusta, layer_mask=None, lod_origin_range_index=-1, list_capacity=0):
        o = np.ascontiguousarray(light_ordinals, np.uint32)
        fr = np.ascontiguousarray(frusta, np.float32).reshape(-1, 6, 6, 4)
        lm = None if layer_mask is None else np.ascontiguousarray(layer_mask, np.uint64)
        self._check(self._lib.b200vis_set_shadow_lights(self._h, len(o), _ptr(o), _ptr(fr), None if lm is None else _ptr(lm),
                                                        int(lod_origin_range_index), int(list_capacity)))

    def set_shadow_items(self, items, list_capacity=0):
        """items: list of dicts(kind, light_row, range, range_view_index, layer_mask, frusta [6,6,4] or [6,4])."""
        arr = (ShadowItem * max(len(items), 1))()
        for i, it in enumerate(items):
            arr[i].kind = it["kind"]; arr[i].light_row = it.get("light_row", 0); arr[i].range = it.get("range", 0.0)
            arr[i].range_view_index = it.get("range_view_index", -1); arr[i].layer_mask = it.get("layer_mask", 1)
            fr = np.zeros((6, 6, 4), np.float32)
            f = np.asarray(it["frusta"], np.float32)
            if f.ndim == 2:
                fr[0] = f
            else:
                fr[:] = f
            arr[i].frusta[:] = fr.reshape(-1).tolist()
        self._check(self._lib.b200vis_set_shadow_items(self._h, len(items), arr, list_capacity))

    def run_shadow_culling(self):
        self._check(self._lib.b200vis_run_shadow_culling(self._h))

    def download_shadow_visible(self, shadow_light, face):
        cnt = C.c_uint32(0)
        self._check(self._lib.b200vis_download_shadow_visible(self._h, shadow_light, face, None, 0, C.byref(cnt)))
        rows = np.zeros(max(cnt.value, 1), np.uint32)
        self._check(self._lib.b200vis_download_shadow_visible(self._h, shadow_light, face, _ptr(rows), len(rows), C.byref(cnt)))
        return rows[:cnt.value]

    # ---- SURVEY 8(f) N4 ----
    def upload_visibility_ranges(self, first, start_end, use_aabb):
        se = np.ascontiguousarray(start_end, np.float32); ua = np.ascontiguousarray(use_aabb, np.uint8)
        self._check(self._lib.b200vis_upload_visibility_ranges(self._h, first, len(ua), _ptr(se), _ptr(ua)))

    def set_visibility_range_views(self, positions):
        p = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
        self._check(self._lib.b200vis_set_visibility_range_views(self._h, len(p), _ptr(p)))

    def download_visibility_ranges(self, first, count):
        out = np.zeros(count, np.uint32)
        self._check(self._lib.b200vis_download_visibility_ranges(self._h, first, count, _ptr(out)))
        return out

    def upload_visibility(self, first, visibility):
        v = np.ascontiguousarray(visibility, np.uint8)
        self._check(self._lib.b200vis_upload_visibility(self._h, first, len(v), _ptr(v)))

    def propagate_visibility(self):
        self._check(self._lib.b200vis_propagate_visibility(self._h))

    def download_inherited_visibility(self, first, count):
        inh, ch = np.zeros(count, np.uint8), np.zeros(count, np.uint8)
        self._check(self._lib.b200vis_download_inherited_visibility(self._h, first, count, _ptr(inh), _ptr(ch)))
        return inh, ch

    # ---- SURVEY 8(f) N2 ----
    def set_cluster_bindings(self, mode, gpu_index_of_light=None):
        """mode: 0 off, 1 storage, 2 uniform (ViewClusterBindings, bevy_pbr/src/cluster/mod.rs:584-800)."""
        m = None if gpu_index_of_light is None else np.ascontiguousarray(gpu_index_of_light, np.uint32)
        self._check(self._lib.b200vis_set_cluster_bindings(self._h, mode, None if m is None else _ptr(m), 0 if m is None else len(m)))
        self._bind_mode = mode

    def download_cluster_bindings(self, view):
        """(offsets_and_counts, index_lists, n_offsets, n_indices) in the mode's wire format."""
        no, ni = C.c_uint32(0), C.c_uint32(0)
        self._check(self._lib.b200vis_download_cluster_bindings(self._h, view, None, 0, None, 0, C.byref(no), C.byref(ni)))
        storage = self._bind_mode == 1
        oc = np.zeros(max(no.value * 8, 1) if storage else 4096, np.uint32)
        il = np.zeros(max(ni.value, 1) if storage else 4096, np.uint32)
        self._check(self._lib.b200vis_download_cluster_bindings(self._h, view, _ptr(oc), len(oc), _ptr(il), len(il), C.byref(no), C.byref(ni)))
        if storage:
            oc, il = oc[:no.value * 8].reshape(-1, 8), il[:ni.value]
        return oc, il, no.value, ni.value

    # ---- SURVEY 8(f) N1 ----
    def enable_visible_diff(self, enabled=True):
        self._check(self._lib.b200vis_enable_visible_diff(self._h, int(bool(enabled))))

    def download_visible_diff(self, view):
        """(added_rows, removed_rows) of `view` against the last frame it was active, both ascending by Entity bits."""
        na, nr = C.c_uint32(0), C.c_uint32(0)
        self._check(self._lib.b200vis_download_visible_diff(self._h, view, None, 0, C.byref(na), None, 0, C.byref(nr)))
        a, r = np.zeros(max(na.value, 1), np.uint32), np.zeros(max(nr.value, 1), np.uint32)
        self._check(self._lib.b200vis_download_visible_diff(self._h, view, _ptr(a), len(a), C.byref(na), _ptr(r), len(r), C.byref(nr)))
        return a[:na.value], r[:nr.value]

    def set_visible_diff_sink(self, rows, counts):
        """Pinned host numpy arrays rows [2, max_views, cap] and counts [max_views, 2]; (None, None) removes the sink."""
        if rows is None:
            self._check(self._lib.b200vis_set_visible_diff_sink(self._h, None, 0, None)); return
        self._check(self._lib.b200vis_set_visible_diff_sink(self._h, _ptr(rows), rows.shape[2], _ptr(counts)))

    def download_visible_by_class(self, view):
        """VisibleEntities::entities of the view as {class k: sorted rows}: the list + class masks, split the way the shim does."""
        rows = self.download_visible(view)
        cls = np.zeros(max(len(rows), 1), np.uint8)
        cnt = C.c_uint32(0)
        self._check(self._lib.b200vis_download_visible_classes(self._h, view, _ptr(cls), len(cls), C.byref(cnt)))
        assert cnt.value == len(rows)
        cls = cls[:len(rows)]
        return {k: rows[(cls >> k) & 1 == 1] for k in range(8) if ((cls >> k) & 1).any()}

    def download_clusters(self, view, capacity=1 << 20):
        offsets = np.zeros(MAX_CLUSTERS + 1, np.uint32); idx = np.zeros(capacity, np.uint32); tot = C.c_uint32(0)
        self._check(self._lib.b200vis_download_clusters(self._h, view, _ptr(offsets), _ptr(idx), capacity, C.byref(tot)))
        return offsets, idx[:tot.value]

    def set_result_sink(self, stats_ptr, visible_rows, cluster_offsets, cluster_indices, visible_classes=None):
        """Pinned host numpy arrays: visible_rows [V, cap], cluster_offsets [V, 4097], cluster_indices [V, cap]; stats_ptr
        is the address of a pinned FrameStats-sized block.  Pass stats_ptr=None to remove the sink."""
        if stats_ptr is None:
            self._check(self._lib.b200vis_set_result_sink(self._h, None)); return
        s = ResultSink()
        s.stats = C.cast(stats_ptr, C.POINTER(FrameStats))
        s.visible_rows = None if visible_rows is None else visible_rows.ctypes.data
        s.visible_capacity = 0 if visible_rows is None else visible_rows.shape[1]
        s.visible_classes = None if visible_classes is None else visible_classes.ctypes.data
        s.cluster_offsets = None if cluster_offsets is None else cluster_offsets.ctypes.data
        s.cluster_indices = None if cluster_indices is None else cluster_indices.ctypes.data
        s.cluster_capacity = 0 if cluster_indices is None else cluster_indices.shape[1]
        self._sink = (s, visible_rows, cluster_offsets, cluster_indices, visible_classes)
        self._check(self._lib.b200vis_set_result_sink(self._h, C.byref(s)))

    def set_column_sinks(self, gt=None, gt_changed_bits=None, view_visibility=None, vv_changed_bits=None):
        """b200vis_set_column_sinks: numpy arrays over (ideally pinned) host memory; gt is [n, 12] or [n, 16] float32.
        All None removes the sinks."""
        if gt is None and gt_changed_bits is None and view_visibility is None and vv_changed_bits is None:
            self._check(self._lib.b200vis_set_column_sinks(self._h, None))
            self._colsink_keep = None
            return
        s = ColumnSinks()
        s.global_transforms = None if gt is None else gt.ctypes.data
        s.gt_stride_floats = 0 if gt is None else gt.shape[1]
        s.gt_changed_bits = None if gt_changed_bits is None else gt_changed_bits.ctypes.data
        s.view_visibility = None if view_visibility is None else view_visibility.ctypes.data
        s.vv_changed_bits = None if vv_changed_bits is None else vv_changed_bits.ctypes.data
        self._colsink_keep = (gt, gt_changed_bits, view_visibility, vv_changed_bits)
        self._check(self._lib.b200vis_set_column_sinks(self._h, C.byref(s)))

    def writeback_columns(self, which=3):
        """which: 1 = GlobalTransform (+ its change bits), 2 = ViewVisibility (+ its change bits), 3 = both."""
        self._check(self._lib.b200vis_writeback_columns_ex(self._h, which))

    def p2p_export(self):
        """CUDA IPC handle (64 bytes) of this rank's gathered buffer."""
        buf = np.zeros(64, np.uint8)
        self._check(self._lib.b200vis_p2p_export(self._h, _ptr(buf)))
        return buf

    def p2p_import(self, handles):
        """handles: uint8 [world, 64], rank-major (as all-gathered by the host)."""
        h = np.ascontiguousarray(handles, np.uint8).reshape(-1, 64)
        self._check(self._lib.b200vis_p2p_import(self._h, _ptr(h)))

    @staticmethod
    def comm_unique_id():
        buf = np.zeros(128, np.uint8)
        rc = load_library().b200vis_comm_unique_id(_ptr(buf))
        if rc:
            raise B200VisError(rc, load_library().b200vis_last_error(None).decode())
        return buf

    def comm_init(self, unique_id):
        uid = _arr(unique_id, np.uint8)
        assert uid.size == 128
        self._check(self._lib.b200vis_comm_init(self._h, _ptr(uid)))

    def cluster_exchange_bytes(self):
        n = C.c_size_t(0)
        self._check(self._lib.b200vis_cluster_exchange_bytes(self._h, C.byref(n)))
        return n.value

    def set_cluster_exchange_buffers(self, send_ptr, recv_ptr):
        self._check(self._lib.b200vis_set_cluster_exchange_buffers(self._h, _vp(send_ptr), _vp(recv_ptr)))
