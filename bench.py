#!/usr/bin/env python
"""bench.py -- entities/s through propagate -> cull -> cluster (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--scaling strong|weak] [--dump-outputs DIR]

A "step" is one frame of the hot path over the synthetic config-#3 scene: 1,000,110 hierarchy entities (3922 complete
binary trees, depth 8, BFS order) + 256 point lights, 4 view frusta, 1920x1080, default ClusterConfig.  Every frame all
3922 roots move (so every GlobalTransform is recomputed and compared, the worst case of the reference's change-driven
path) and the cameras rotate.

  value         device-resident inputs: the per-frame root Transforms and frame constants already sit in HBM; frames are
                enqueued back to back (the tail of frame f overlaps the tile pass of frame f+1: pipelined THROUGHPUT, not the
                latency of one frame -- a live frame with the Clusters feedback loop is the e2e figure); CUDA events on the
                launching stream, max over ranks.
  e2e           one C-ABI call per frame (b200vis_step) with HOST buffers: changed Transforms from pinned host memory,
                per-view constants recomputed on the host with last frame's feedback, and EVERY result written back to host
                memory inside the timed region: frame stats, sorted visible lists, cluster lists, every changed
                GlobalTransform in glam's 64-byte Affine3A layout, the ViewVisibility bytes and both change-flag bit sets
                (b200vis_set_column_sinks).  `e2e_resident` = the same without the column write-back (round 1's figure),
                `e2e_sparse` = the reference bench's own mutation pattern (8 roots per frame, propagate.rs:115-128).
  N > 1         --scaling strong (default; what BASELINE.json's metric quotes): the SAME 1M / 256 scene split by whole-tree
                row ranges; --scaling weak: every rank owns a 1M / 256 shard.  One exchange per frame: an all-gather of the
                ranks' light-record blocks (28 B per light: this frame's position + ViewVisibility, range, layers), after
                which every rank runs the one-launch cluster stage over all lights.  B200VIS_EXCHANGE=p2p sends the same
                blocks as peer stores over NVLink; B200VIS_EXCHANGE_WHAT=slabs exchanges the cluster x light bit slabs
                instead (the path for light counts beyond the cluster kernel's shared memory).
  parity        outside the timed regions the frame that follows each timed loop is checked bit for bit against the CPU
                oracle (GlobalTransform bits, both change columns, ViewVisibility, sorted visible lists, cluster CSR, column
                write-back) on every rank: `parity_checked`.
  outputs       --dump-outputs DIR writes the results of the last step of the device-resident timed loop as .npy files
                (dump_outputs); the inputs are seeded, so two builds run with the same arguments compute the same frame.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The driver parses ONE JSON line from stdout: keep the real stdout for it and send everything else
# (NCCL's version banner, library chatter) to stderr.
REAL_STDOUT = os.dup(1)
os.dup2(2, 1)
sys.stdout = sys.stderr

METRIC = "entities/s propagate+cull+cluster @1M ents/256 lights"
N_TREES, LEVELS, N_LIGHTS = 3922, 8, 256
PER_TREE = (1 << LEVELS) - 1
ALGO_BYTES_PER_ENTITY = 119      # SURVEY.md 8(d): fused propagate->cull, compact SoA
EXTRA_BYTES_NOTE = "exact set_if_neq also reads the old GlobalTransform (+48 B/entity of compulsory traffic, not counted)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--trees", type=int, default=N_TREES)
    ap.add_argument("--lights", type=int, default=N_LIGHTS)
    ap.add_argument("--cpu-frames", type=int, default=40, help="frames of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-next-rows", action="store_true", help="skip the SURVEY 8(f) row measurements (N1, N2, N4)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle checks (they run outside the timed regions)")
    ap.add_argument("--no-secondary", action="store_true", help="N > 1: skip the other scaling mode's short measurement")
    ap.add_argument("--print-config", action="store_true", help="print the `config` object of this command line and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy (b200 arm)")
    return ap.parse_args()


def workload_config(args):
    """The `config` object: a function of the command line only, identical for both arms."""
    n_gpus = max(args.gpus, 1)
    weak = args.scaling == "weak" and n_gpus > 1
    ents = args.trees * PER_TREE + args.lights
    total_e, total_l = (ents * n_gpus, args.lights * n_gpus) if weak else (ents, args.lights)
    return {"workload": (f"config#3 forest {args.trees}x{PER_TREE} (BFS, depth {LEVELS}) + {args.lights} point lights"
                         + (" per GPU" if weak else "") + ", 4 views 1920x1080, default ClusterConfig, all roots move every frame"),
            "scaling": "weak" if weak else "strong", "entities_total": total_e, "lights_total": total_l, "views": 4,
            "l2": "working set 167 MB/frame > 126 MB L2 at 1M entities per GPU (inputs larger than L2, no flush)"}


# ---------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md): sampled DURING the timed region
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [s for t, s in self.samples if t0 - 0.05 <= t <= t1 + 0.15] or [s for _, s in self.samples]
        mhz, mx, reasons = [], None, set()
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 6:
                continue
            try:
                mhz.append(float(p[0])); mx = float(p[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(mhz)) if mhz else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(mhz)}


def emit(line):
    os.write(REAL_STDOUT, (json.dumps(line) + "\n").encode())


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's multithreaded restatement on the host cores
# ---------------------------------------------------------------------------------------------
def physical_cores():
    """Threads for the CPU arm: physical cores this process may use -- affinity mask, SMT siblings counted once, and the
    container's CPU quota (cgroup cpu.max), because threads beyond the quota are throttled, not run."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or aff
    except Exception:
        phys = aff
    n = max(1, min(aff, phys))
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = max(1, min(n, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = max(1, min(n, q // period))
            break
        except Exception:
            continue
    return n


class CpuArm:
    """propagate -> cull -> cluster of the same workload with the multithreaded CPU restatement (oracle/bevy_oracle_mt.c):
    OpenMP over roots / contiguous row ranges and a serial merge + sort of the visible lists, as the reference does.
    Threads = physical cores (fixed, pinned with OMP_PROC_BIND=close / OMP_PLACES=cores), stated in the output."""

    def __init__(self, scene):
        os.environ.setdefault("OMP_PROC_BIND", "close")
        os.environ.setdefault("OMP_PLACES", "cores")
        os.environ.setdefault("OMP_WAIT_POLICY", "active")
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle as orc            # bench.py executes oracle/ only as the measured CPU baseline and as the checker
        from bevy_b200 import scenes
        from parity import OracleWorld
        self.orc, self.scenes, self.scene = orc, scenes, scene
        self.world = OracleWorld(scene, static_opt=True)
        self.frame_no = 0
        # thread count: physical cores (quota-aware); on a shared or quota-limited host fewer threads can be faster (threads
        # beyond the CPUs actually granted are throttled, and the merge + sort of the visible lists is serial), so a few
        # fixed fractions are tried on warm frames and the best median is kept -- the figure reported is that one
        cores = physical_cores()
        self.frame(); self.frame()                    # first touch / page faults
        best = None
        for nt in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 16), min(cores, 8)}, reverse=True):
            orc.lib_mt().orc_mt_set_threads(nt)
            self.frame()
            med = float(np.median([self.frame() for _ in range(3)]))
            if best is None or med < best[0]:
                best = (med, nt)
        self.threads = best[1]
        self.calibration = f"{self.threads} of {cores} cores (best median of 3 warm frames among fixed fractions of the core count)"
        orc.lib_mt().orc_mt_set_threads(self.threads)

    def frame(self):
        f = self.frame_no; self.frame_no += 1
        sc = self.scene
        if f > 0:
            self.scenes.advance_cameras(sc)
            rows, _ = self.scenes.mutate_roots(sc, f)
            self.world.tchanged[rows] = 1
        planes = np.stack([self.orc.compute_frustum(self.orc.perspective(c.fov, c.aspect, c.near), c.gt, c.far) for c in sc.cameras])
        t0 = time.perf_counter()
        self.world.frame(planes, cluster=True, mt=True)
        return time.perf_counter() - t0

    def run(self, steps, warmup):
        for _ in range(warmup):
            self.frame()
        return np.array([self.frame() for _ in range(steps)])


def cpu_summary(times, n, threads, what, calibration=""):
    med = float(np.median(times))
    return {"value": n / med, "unit": "entities/s", "cores": threads, "kind": "port",
            "ms_per_step_median": med * 1e3, "ms_per_step_min": float(times.min()) * 1e3, "ms_per_step_max": float(times.max()) * 1e3,
            "threads": calibration,
            "sample": what + "; OpenMP, pinned (OMP_PROC_BIND=close, OMP_PLACES=cores); Rust toolchain "
                             "absent: C restatement of the reference algorithm (oracle/bevy_oracle_mt.c), not Bevy itself"}


def run_reference(args):
    if args.dump_outputs:
        raise SystemExit("--dump-outputs writes the b200 arm's results; the reference arm has none to write")
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from bevy_b200 import scenes
    cfg = workload_config(args)
    # the CPU has no per-GPU shards: it runs the whole workload the b200 arm's N GPUs run together (weak: N shards' worth)
    n_shards = args.gpus if cfg["scaling"] == "weak" else 1
    scene = scenes.forest(args.trees * n_shards, LEVELS, args.lights * n_shards)
    arm = CpuArm(scene)
    K, W = max(args.steps, 1), max(args.warmup, 0)
    # a step is one full frame; should K of them not fit into a few minutes, a step becomes a bounded sample of the frame
    # (the first S trees), sized from two probe frames
    probe = max(arm.frame(), arm.frame())
    budget = 240.0
    sample_note = f"{K} full frames of the {scene.n}-entity workload after {W} warm-up frames"
    if probe * (K + W) > budget:
        frac = budget / (probe * (K + W))
        trees = max(64, int(args.trees * n_shards * frac))
        scene = scenes.forest(trees, LEVELS, args.lights * n_shards)
        arm = CpuArm(scene)
        sample_note = (f"{K} frames of a bounded sample ({trees} of {args.trees * n_shards} trees, all lights) after {W} warm-up frames: "
                       f"a full frame takes {probe * 1e3:.1f} ms here")
    times = arm.run(K, W)
    n = scene.n
    cb = cpu_summary(times, n, arm.threads, sample_note, arm.calibration)
    val = cb["value"]
    emit({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "entities/s", "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": cb["ms_per_step_median"], "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "entities/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
class Rig:
    """One rank's context + the precomputed animation + pinned result buffers for one scaling mode."""

    def __init__(self, args, torch, dist, bb, scenes, parallel, scaling, world, rank, local_rank, dev, stream):
        self.args, self.torch, self.dist, self.bb, self.scenes = args, torch, dist, bb, scenes
        self.world, self.rank, self.dev, self.stream = world, rank, dev, stream
        self.scaling = scaling
        if scaling == "weak" or world == 1:
            # every rank owns one shard: its own trees (seeded per rank) and its own lights; cameras are replicated
            self.full = None
            self.scene = scenes.forest(args.trees, LEVELS, args.lights, seed=42 + (rank if world > 1 else 0))
            self.rows_of_full = None
            self.light_ranges = [(r * args.lights, (r + 1) * args.lights) for r in range(world)]
            max_lights = args.lights
        else:
            # strong: the same scene for every N, split by whole-tree row ranges; the lights shard with their rows
            self.full = scenes.forest(args.trees, LEVELS, args.lights, seed=42)
            self.scene, self.rows_of_full, _ = parallel.shard_scene(self.full, rank, world, PER_TREE)
            self.light_ranges = parallel.shard_bounds(args.lights, world)
            max_lights = max(hi - lo for lo, hi in self.light_ranges)
        sc = self.scene
        self.n, self.V = sc.n, len(sc.cameras)
        self.pipe = bb.VisibilityPipeline(sc, device=local_rank, world_size=world, rank=rank, max_lights=max(max_lights, 1))
        self.ctx = ctx = self.pipe.ctx
        ctx.set_stream(stream.cuda_stream)
        self.max_lights_cap = ((max(1, max_lights) + 31) // 32) * 32
        if world > 1:
            exchange = os.environ.get("B200VIS_EXCHANGE", "nccl")
            if exchange == "p2p":
                mine = torch.from_numpy(ctx.p2p_export()).to(dev)
                handles = torch.zeros((world, 64), dtype=torch.uint8, device=dev)
                dist.all_gather_into_tensor(handles.view(-1), mine)
                ctx.p2p_import(handles.cpu().numpy())
                dist.barrier()
            else:
                # built-in exchange: the library issues the one ncclAllGather of the cluster slabs itself (the NCCL the process
                # already loaded for torch.distributed); the 128-byte unique id travels over torch.distributed
                uid = torch.zeros(128, dtype=torch.uint8, device=dev)
                if rank == 0:
                    uid.copy_(torch.from_numpy(bb.Context.comm_unique_id()))
                dist.broadcast(uid, 0)
                ctx.comm_init(uid.cpu().numpy())
            self.exchange = exchange
        else:
            self.exchange = "none"
        # ---- the animation: per-frame root Transforms (pinned host + device copies) and camera poses ------------
        self.WIN = WIN = 64           # recorded animation window; frames cycle through it (results change every frame)
        self.n_roots = n_roots = len(sc.roots)
        self.rows_h = torch.from_numpy(sc.roots.astype(np.int32)).pin_memory()
        self.trs_h = torch.empty((2 * WIN, max(n_roots, 1), 10), dtype=torch.float32).pin_memory()
        self.cam_frames = []
        for f in range(2 * WIN):
            scenes.advance_cameras(sc)
            if n_roots:
                _, trs = scenes.mutate_roots(sc, f + 1)
                self.trs_h[f, :n_roots].copy_(torch.from_numpy(trs))
            self.cam_frames.append([(c.gt.copy(), c.quat.copy()) for c in sc.cameras])
        self.rows_d = self.rows_h.to(dev)
        self.trs_d = self.trs_h.to(dev)
        self.cam_descs = []
        for f in range(2 * WIN):
            arr = (bb.CameraDesc * self.V)()
            for v, (cam, (gt, q)) in enumerate(zip(sc.cameras, self.cam_frames[f])):
                arr[v].global_transform[:] = gt.tolist()
                arr[v].fov_y, arr[v].aspect, arr[v].near_z, arr[v].far_z = cam.fov, cam.aspect, cam.near, cam.far
                arr[v].layer_mask, arr[v].flags, arr[v].range_view_index = 1, bb.VIEW_ACTIVE, -1
            self.cam_descs.append(arr)
        # ---- pinned host buffers the results land in (what a shim would hand to VisibleEntities / Clusters / the columns)
        n, V = self.n, self.V
        pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory()      # noqa: E731
        self.vis_h = pin((V, max(n, 1)), torch.int32).numpy().view(np.uint32)
        self.coff_h = pin((V, 4097), torch.int32).numpy().view(np.uint32)
        self.cidx_h = pin((V, 1 << 18), torch.int32).numpy().view(np.uint32)
        self.stats_t = pin(ctypes.sizeof(bb.FrameStats), torch.uint8)
        self.stats = bb.FrameStats.from_address(self.stats_t.data_ptr())
        self.gt_h = pin((max(n, 1), 16), torch.float32).numpy()                 # the GlobalTransform column, glam Affine3A layout
        self.gt_h[:] = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0], np.float32)
        W32 = (n + 31) // 32
        self.gbits_h = pin(max(W32, 1), torch.int32).numpy().view(np.uint32)
        self.vbits_h = pin(max(W32, 1), torch.int32).numpy().view(np.uint32)
        self.vv_h = pin(max(n, 1), torch.uint8).numpy()

    def set_cameras(self, f):
        for c, (gt, q) in zip(self.scene.cameras, self.cam_frames[f]):
            c.gt, c.quat = gt, q

    def sinks(self, on, columns):
        c = self.ctx
        if on:
            c.set_result_sink(self.stats_t.data_ptr(), self.vis_h, self.coff_h, self.cidx_h)
        else:
            c.set_result_sink(None, None, None, None)
        if on and columns:
            c.set_column_sinks(self.gt_h, self.gbits_h, self.vv_h, self.vbits_h)
        else:
            c.set_column_sinks()

    def e2e_step(self, f, writeback=True, n_changed=None):
        # ONE call per frame through the C ABI: upload changed Transforms (pinned host -> HBM), host-side per-view maths with
        # last frame's feedback, all kernels (+ the one exchange when N > 1), the GPU writes every result into pinned host
        # memory, one sync
        k = self.n_roots if n_changed is None else min(n_changed, self.n_roots)
        self.ctx.step(k, self.rows_h.data_ptr(), self.trs_h[f].data_ptr(), self.cam_descs[f], self.V, self.pipe.cluster_config,
                      wait=True, writeback=writeback)

    def d2h_bytes(self, writeback):
        st = self.stats
        nb = ctypes.sizeof(st)
        for v in range(self.V):
            cv = self.ctx.cluster_dims(v)
            nb += 4 * st.visible_count[v] + 4 * (cv + 1) + 4 * st.cluster_index_count[v]
        if writeback:
            nb += 64 * st.gt_changed_count + self.n + 2 * 4 * ((self.n + 31) // 32)
        return nb

    def value_setup(self):
        """Run one animation window once with the feedback loop closed and record each frame's constants (views, cluster
        tables) as a blob in HBM, so that the timed replay has every input resident."""
        ctx, pipe = self.ctx, self.pipe
        self.slots = []
        for i in range(self.WIN):
            f = self.WIN + i
            self.set_cameras(f)
            ctx.upload_transforms_scattered_raw(self.n_roots, self.rows_d.data_ptr(), self.trs_d[f].data_ptr())
            pipe.update_views_fast()
            self.slots.append(ctx.record_frame_constants())
            ctx.run(self.bb.STAGE_ALL)
            pipe.read_feedback()

    def value_step(self, i):
        # device-resident inputs only: this frame's root Transforms and constants are already in HBM
        i %= self.WIN
        self.ctx.upload_transforms_scattered_raw(self.n_roots, self.rows_d.data_ptr(), self.trs_d[self.WIN + i].data_ptr())
        self.ctx.use_recorded_frame_constants(self.slots[i])
        self.ctx.run(self.bb.STAGE_ALL)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, step, K, W, first=0):
        """W warm-up + K timed calls of step(frame); returns (device ms by CUDA events on the launching stream, wall s)."""
        torch = self.torch
        for f in range(W):
            step(first + f)
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(self.stream)
        for f in range(W, W + K):
            step(first + f)
        self.enqueue_s = time.perf_counter() - t0      # host time to enqueue the K steps (no synchronisation inside for `value`)
        self.ctx.join()                  # the last frame's tail (side stream) belongs to the timed region
        ev1.record(self.stream)
        self.barrier()
        return ev0.elapsed_time(ev1), time.perf_counter() - t0

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    # ---- parity: the frame after a timed loop, checked bit for bit against the CPU oracle ---------------------------------
    def parity_check(self, f, mode):
        """Takes the device's current state as the oracle's start state, runs frame `f` on both, compares every output of
        this rank's shard; the cluster lists are compared against the oracle's assignment of ALL ranks' lights."""
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle as orc
        from parity import OracleWorld
        torch, dist, ctx, sc, n, V = self.torch, self.dist, self.ctx, self.scene, self.n, self.V
        world_o = OracleWorld(sc, static_opt=True)
        gt0, _ = ctx.download_global_transforms(0, n)
        vv0, _ = ctx.download_view_visibility(0, n)
        world_o.gt[:], world_o.vv[:] = gt0, vv0
        world_o.tchanged[:] = 0
        prev = ctx.download_frame_stats()
        fb = [(float(prev.cluster_farthest_z[v]), int(prev.cluster_index_count[v])) for v in range(V)]
        # inputs of frame f on the oracle side
        f = f % self.WIN if mode == "e2e" else self.WIN + f % self.WIN
        trs = self.trs_h[f, :self.n_roots].numpy()
        sc.trs[sc.roots] = trs
        world_o.tchanged[sc.roots] = 1
        self.set_cameras(f)
        planes = np.stack([orc.compute_frustum(orc.perspective(c.fov, c.aspect, c.near), c.gt, c.far) for c in sc.cameras])
        gt_changed, vv_changed, lists, _ = world_o.frame(planes, cluster=False)
        # ... and on the device, through the same call the timed loop used
        if mode == "e2e":
            mirror_before = self.gt_h.copy()
            self.e2e_step(f, writeback=True)
            ctx.synchronize()
        else:
            self.value_step(f - self.WIN)
            ctx.join(); ctx.synchronize()
        errs = []
        gt, ch = ctx.download_global_transforms(0, n)
        if not (gt.view(np.uint32) == world_o.gt.view(np.uint32)).all():
            errs.append("GlobalTransform bits")
        if not (ch == gt_changed).all():
            errs.append("Changed<GlobalTransform>")
        vv, vch = ctx.download_view_visibility(0, n)
        if not (vv == world_o.vv).all():
            errs.append("ViewVisibility")
        if not (vch == vv_changed).all():
            errs.append("Changed<ViewVisibility>")
        for v in range(V):
            got = ctx.download_visible(v)
            if len(got) != len(lists[v]) or not (got == lists[v]).all():
                errs.append(f"visible list view {v}")
        if mode == "e2e":       # the column write-back: the host mirror equals the device column; untouched rows kept their bytes
            gt16, _ = ctx.download_global_transforms(0, n, stride=16)
            unpack = lambda b: np.unpackbits(b.view(np.uint8), bitorder="little")[:n]     # noqa: E731
            if not (self.gt_h[:n].view(np.uint32) == gt16.view(np.uint32)).all():
                errs.append("write-back: GlobalTransform column")
            if not (self.gt_h[:n][ch == 0].view(np.uint32) == mirror_before[:n][ch == 0].view(np.uint32)).all():
                errs.append("write-back: unchanged rows were written")
            if not (unpack(self.gbits_h) == ch).all() or not (unpack(self.vbits_h) == vch).all():
                errs.append("write-back: change bits")
            if not (self.vv_h[:n] == vv).all():
                errs.append("write-back: ViewVisibility column")
            for v in range(V):
                c = self.stats.visible_count[v]
                if c != len(lists[v]) or not (self.vis_h[v, :c] == lists[v]).all():
                    errs.append(f"sink: visible list view {v}")
        # clusters: every rank's visible lights, in global light order
        lr = sc.light_row
        mine = np.concatenate([world_o.gt[lr, 9:12], sc.light_range[:, None], (world_o.vv[lr] & 1)[:, None].astype(np.float32)], 1) \
            .astype(np.float32) if len(lr) else np.zeros((0, 5), np.float32)
        if self.world > 1:
            pad = np.zeros((self.max_lights_cap, 5), np.float32); pad[:len(mine)] = mine
            cnt = torch.tensor([len(mine)], device=self.dev)
            buf = torch.from_numpy(pad).to(self.dev)
            allb = torch.zeros((self.world,) + tuple(buf.shape), device=self.dev)
            allc = torch.zeros(self.world, dtype=cnt.dtype, device=self.dev)
            dist.all_gather_into_tensor(allb.view(-1), buf.view(-1)); dist.all_gather_into_tensor(allc, cnt)
            allb, allc = allb.cpu().numpy(), allc.cpu().numpy()
            lights_all = np.concatenate([allb[r, :allc[r]] for r in range(self.world)])
        else:
            lights_all = mine
        vis_idx = np.nonzero(lights_all[:, 4] > 0)[0]
        lights = np.ascontiguousarray(lights_all[vis_idx, :4])
        stats = ctx.download_frame_stats()
        from bevy_b200 import parallel
        for v, cam in enumerate(sc.cameras):
            cfv = orc.perspective(cam.fov, cam.aspect, cam.near)
            vin = orc.default_cluster_view_in(cam.gt, cfv, planes[v], screen=sc.screen, view_layers=1,
                                              last_farthest_z=fb[v][0], last_index_count=fb[v][1])
            out, offsets, idx, _ = orc.assign_lights_to_clusters(vin, lights, None)
            goff, gidx = ctx.download_clusters(v)
            nc = out.dims[0] * out.dims[1] * out.dims[2]
            want = vis_idx[idx]
            glob = parallel.global_light_ordinal(gidx, self.max_lights_cap, self.light_ranges) if self.world > 1 else gidx
            if ctx.cluster_dims(v) != nc or not (goff[:nc + 1] == offsets).all() or len(glob) != len(want) or not (glob == want).all():
                errs.append(f"cluster lists view {v}")
            if stats.cluster_index_count[v] != out.total_index_count or \
                    np.float32(stats.cluster_farthest_z[v]).view(np.uint32) != np.float32(out.farthest_z).view(np.uint32):
                errs.append(f"cluster feedback view {v}")
        return errs

    def close(self):
        self.pipe.close()


def measure_pcie(torch, dev, stream):
    """Achievable host<->device copy rates of this box (pinned memory, copy engine): what the write-back is measured against."""
    n = 256 << 20
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    out = {}
    for name, (dst, src) in (("d2h_gbs", (h, d)), ("h2d_gbs", (d, h))):
        best = 0.0
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); dst.copy_(src, non_blocking=True); e1.record(stream)
            torch.cuda.synchronize()
            best = max(best, n / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        out[name] = best
    return out


DUMP_ROWS = 1 << 18             # per-row columns: a seeded sample of this many rows (every row when there are fewer)
DUMP_LIST_ENTRIES = 1 << 21     # visible lists, and again cluster index lists: at most this many entries over all views
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, ctx, n, V):
    """Writes what the last step computed, as a caller of the device-resident path downloads it: GlobalTransforms, both
    change columns, ViewVisibility, the sorted visible lists, the cluster lists and the frame stats.  Long outputs are
    reduced to a fixed seeded sample (the sampled row ids go to rows.npy), so that the files stay below DUMP_MAX_BYTES at
    any scene size and two builds run with the same arguments can be compared file for file."""
    def sample(count, cap, seed):
        if count <= cap:
            return np.arange(count)
        return np.sort(np.random.default_rng(seed).choice(count, cap, replace=False))

    rows = sample(n, DUMP_ROWS, 0)
    gt, gt_changed = ctx.download_global_transforms(0, n)
    vv, vv_changed = ctx.download_view_visibility(0, n)
    stats = ctx.download_frame_stats()
    out = {"rows": rows.astype(np.float64), "global_transform": gt[rows],
           "global_transform_changed": gt_changed[rows].astype(np.float32),
           "view_visibility": vv[rows].astype(np.float32), "view_visibility_changed": vv_changed[rows].astype(np.float32),
           "visible_count": np.array(stats.visible_count[:V], np.float64),
           "cluster_index_count": np.array(stats.cluster_index_count[:V], np.float64),
           "cluster_farthest_z": np.array(stats.cluster_farthest_z[:V], np.float32),
           "changed_count": np.array([stats.gt_changed_count, stats.vv_changed_count], np.float64)}
    for v in range(V):
        vis = ctx.download_visible(v)
        out[f"visible_rows_view{v}"] = vis[sample(len(vis), DUMP_LIST_ENTRIES // V, 1 + v)].astype(np.float64)
        offsets, idx = ctx.download_clusters(v)
        out[f"cluster_offsets_view{v}"] = offsets[:ctx.cluster_dims(v) + 1].astype(np.float64)
        out[f"cluster_indices_view{v}"] = idx[sample(len(idx), DUMP_LIST_ENTRIES // V, 1 + V + v)].astype(np.float64)
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_next_rows(torch, bb, rig, tile_ms, expand_ms, cluster_ms, e2e_resident_ms, W):
    """Cost of the SURVEY.md 8(f) rows on the bench workload (1 GPU): stage times with the row switched on against the
    base numbers measured above (same CUDA-event stage timers), plus the e2e frame when the shim takes the added /
    removed lists (N1) instead of the full visible lists."""
    ctx, pipe, scene, stream = rig.ctx, rig.pipe, rig.scene, rig.stream
    n, V, F, WIN = scene.n, len(scene.cameras), 100, rig.WIN
    out = {}

    def staged(frames=F, step=None):
        step = step or rig.value_step
        ctx.set_profiling(True)
        for i in range(frames):
            step(i)
        t, e, c, nf = ctx.collect_stage_times_ms()
        ctx.set_profiling(False)
        return t / nf, e / nf, c / nf

    # N1: device-side added / removed lists
    ctx.enable_visible_diff(True)
    for i in range(W):
        rig.value_step(i)
    _, e_ms, _ = staged()
    diff_counts = [tuple(len(x) for x in ctx.download_visible_diff(v)) for v in range(V)]
    ctx.use_recorded_frame_constants(None)
    cap = 1 << 16
    rows_h = torch.zeros((2, V, cap), dtype=torch.int32).pin_memory()
    counts_h = torch.zeros((V, 2), dtype=torch.int32).pin_memory()
    ctx.set_visible_diff_sink(rows_h.numpy().view(np.uint32), counts_h.numpy().view(np.uint32))
    ctx.set_result_sink(rig.stats_t.data_ptr(), None, rig.coff_h, rig.cidx_h)      # full visible lists stay on the device
    for f in range(W):
        rig.e2e_step(f % WIN, writeback=False)
    torch.cuda.synchronize()
    KD = 300
    t0 = time.perf_counter()
    for f in range(W, W + KD):
        rig.e2e_step(f % WIN, writeback=False)
    torch.cuda.synchronize()
    e2e_diff_ms = (time.perf_counter() - t0) * 1e3 / KD
    d2h = int(np.mean([4 * (counts_h[v, 0].item() + counts_h[v, 1].item()) for v in range(V)]) * V)
    ctx.set_result_sink(None, None, None, None)
    ctx.set_visible_diff_sink(None, None)
    ctx.enable_visible_diff(False)
    out["N1_visible_diff"] = {"expand_plus_diff_ms": e_ms, "expand_only_ms": expand_ms,
                              "added_removed_last_frame": diff_counts,
                              "e2e_resident_ms_per_step_with_diff_sink": e2e_diff_ms, "e2e_resident_ms_per_step_full_lists": e2e_resident_ms,
                              "visible_d2h_bytes_per_step_with_diff_sink": d2h}

    # N2: ViewClusterBindings wire format straight from the cluster CSR
    for mode, name in ((1, "storage"), (2, "uniform")):
        ctx.set_cluster_bindings(mode)
        _, _, c_ms = staged()
        oc, il, no, ni = ctx.download_cluster_bindings(0)
        out[f"N2_cluster_bindings_{name}"] = {"cluster_ms": c_ms, "cluster_only_ms": cluster_ms, "n_offsets_view0": no, "n_indices_view0": ni}
    ctx.set_cluster_bindings(0)

    # N3: shadow-view culling, 16 of the lights cast shadows, every tree mesh is a caster (CUDA events on the launching stream)
    from bevy_b200 import abi as _abi
    S = min(16, len(scene.light_row))
    if S:
        caster = np.ones(n, np.uint8); caster[scene.light_row] = 0
        ctx.upload_shadow_casters(0, caster)
        for i in range(W):
            rig.value_step(i)                                  # the view sets are recorded from here on
        ctx.join()
        ords = np.sort(np.argsort(-scene.light_range)[:S]).astype(np.uint32)     # the S lights with the largest range
        frusta = np.zeros((S, 6, 6, 4), np.float32)
        for i, o in enumerate(ords):
            gt, _ = ctx.download_global_transforms(int(scene.light_row[o]), 1, want_changed=False)
            frusta[i] = _abi.host_point_light_frusta(gt[0], float(scene.light_range[o]), 0.1)
        ctx.set_shadow_lights(ords, frusta, None, -1, 1 << 16)
        ctx.run_shadow_culling()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        torch.cuda.synchronize()
        reps = 20
        ev[0].record(stream)
        for _ in range(reps):
            ctx.run_shadow_culling()
        ev[1].record(stream)
        torch.cuda.synchronize()
        sh_ms = ev[0].elapsed_time(ev[1]) / reps
        pairs = sum(len(ctx.download_shadow_visible(i, f)) for i in range(S) for f in range(6))
        out["N3_point_light_shadow_culling"] = {
            "ms": sh_ms, "shadow_lights": S, "caster_rows": int(caster.sum()), "row_light_pairs_per_s": S * float(caster.sum()) / (sh_ms * 1e-3),
            "visible_row_face_pairs": int(pairs)}
        ctx.enable_visible_diff(False)

    # N4b: visibility_propagate_system over all rows (CUDA events on the launching stream)
    rng = np.random.default_rng(7)
    vis = rng.choice([0, 0, 0, 1, 2], n).astype(np.uint8)
    ctx.upload_visibility(0, vis)
    ctx.propagate_visibility()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    reps = 50
    ev[0].record(stream)
    for _ in range(reps):
        ctx.propagate_visibility()
    ev[1].record(stream)
    torch.cuda.synchronize()
    vp_ms = ev[0].elapsed_time(ev[1]) / reps
    inh, _ = ctx.download_inherited_visibility(0, n)
    out["N4_visibility_propagate"] = {"ms": vp_ms, "algorithmic_bytes_per_entity": 7,
                                      "achieved_GBps": n * 7 / (vp_ms * 1e-3) / 1e9, "inherited_visible_rows": int(inh.sum())}
    ctx.upload_visibility(0, np.zeros(n, np.uint8)); ctx.propagate_visibility()      # everything visible again

    # N4a: check_visibility_ranges inside the cull phase, VisibilityRange on EVERY row, range views = the 4 cameras
    se = np.stack([np.zeros(n, np.float32), np.full(n, 700.0, np.float32)], 1)
    ctx.upload_visibility_ranges(0, se, np.ones(n, np.uint8))
    flags = (scene.flags | bb.F_HAS_VIS_RANGE).astype(np.uint8)
    ctx.upload_bounds(0, scene.bounds, flags, scene.class_mask, scene.layer_mask, None)
    ctx.set_visibility_range_views(np.stack([np.asarray(c.gt, np.float32)[9:12] for c in scene.cameras]))
    ctx.use_recorded_frame_constants(None)
    scene.view_range_index = list(range(V))  # each culled view reads its own bit of the range mask

    def live_step(i):
        f = WIN + i % WIN
        rig.set_cameras(f)
        ctx.upload_transforms_scattered_raw(rig.n_roots, rig.rows_d.data_ptr(), rig.trs_d[f].data_ptr())
        pipe.update_views_fast()
        ctx.run(bb.STAGE_ALL)

    for i in range(W):
        live_step(i)
    t_ms, _, _ = staged(step=live_step)
    masks = ctx.download_visibility_ranges(0, n)
    out["N4_visibility_ranges"] = {"tile_ms_all_rows_ranged": t_ms, "tile_ms_base": tile_ms, "rows_in_range_of_view0": int((masks & 1).sum())}
    return out


def main():
    args = parse_args()
    if args.print_config:
        return emit(workload_config(args))
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import bevy_b200 as bb
    from bevy_b200 import abi, parallel, scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"WORLD_SIZE {world} != --gpus {args.gpus}"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: libb200vis has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, max(args.warmup, 3)
    # Everything (library kernels, copies, NCCL, timing events) runs on ONE explicit non-default stream: torch's
    # default stream has handle 0, which b200vis_set_stream reads as "use the context's own stream".
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    cfg = workload_config(args)
    scaling = cfg["scaling"]
    rig = Rig(args, torch, dist, bb, scenes, parallel, scaling, world, rank, local_rank, dev, stream)
    ctx, n, V = rig.ctx, rig.n, rig.V
    total_entities = cfg["entities_total"]
    parity = {"checked": False, "errors": []}

    # first frame: everything is "Added"; run it once so steady state starts from real GlobalTransforms
    ctx.run(bb.STAGE_ALL)
    rig.pipe.read_feedback()
    # the host columns start as a copy of the device's (spawn-time state); from here on only the write-back touches them
    rig.gt_h[:n] = ctx.download_global_transforms(0, n, stride=16, want_changed=False)[0]
    rig.vv_h[:n] = ctx.download_view_visibility(0, n)[0]
    pcie = measure_pcie(torch, dev, stream) if rank == 0 else None

    # ---- pass A: e2e through the plugin API with host buffers, every result written back ----------------------------------
    WIN = rig.WIN
    rig.sinks(True, True)
    launches0 = abi.kernel_launch_count()
    e2e_dev_ms, e2e_wall = rig.timed(lambda f: rig.e2e_step(f % WIN, True), K, W)
    e2e_launches = (abi.kernel_launch_count() - launches0) / (K + W)
    e2e_sec = max(e2e_wall, e2e_dev_ms / 1e3)
    e2e_d2h = rig.d2h_bytes(True)
    e2e_h2d = rig.n_roots * 44 + 8192         # root TRS + row ids + the frame-constant blob (upper bound of its used part)
    gt_changed_e2e = int(rig.stats.gt_changed_count)
    visible_pairs = sum(rig.stats.visible_count[v] for v in range(V))
    cluster_indices = sum(rig.stats.cluster_index_count[v] for v in range(V))
    if not args.no_parity:
        parity["errors"] += [f"e2e: {e}" for e in rig.parity_check(W + K, "e2e")]
    # where the e2e frame goes on the device (CUDA events around the stages, a few extra frames, not part of the timing)
    ctx.set_profiling(True)
    for f in range(40):
        rig.e2e_step((W + K + 1 + f) % WIN, True)
    pt, pe_, pc, pn = ctx.collect_stage_times_ms()
    ctx.set_profiling(False)
    e2e_breakdown = {"tile_ms": pt / max(pn, 1) * 2, "expand_ms": pe_ / max(pn, 1) * 2, "cluster_ms": pc / max(pn, 1) * 2}
    # A2: the same without the column write-back (round 1's e2e), A3: the reference bench's sparse mutation pattern
    K2 = max(50, min(K, 500))
    rig.sinks(True, False)
    res_dev_ms, res_wall = rig.timed(lambda f: rig.e2e_step(f % WIN, False), K2, W)
    res_d2h = rig.d2h_bytes(False)
    rig.sinks(True, True)
    sp_dev_ms, sp_wall = rig.timed(lambda f: rig.e2e_step(f % WIN, True, n_changed=8), K2, W)
    sp_d2h = rig.d2h_bytes(True)
    sp_changed = int(rig.stats.gt_changed_count)
    rig.sinks(False, False)
    # all roots move again before the device-resident pass
    rig.e2e_step(0, False)

    # ---- pass B: device-resident replay ---------------------------------------------------------------------------------
    rig.value_setup()
    sampler = ClockSampler(local_rank)
    for i in range(W):
        rig.value_step(i)
    rig.barrier()
    sampler.start()
    ts0 = time.time()
    launches0 = abi.kernel_launch_count()
    dev_ms, _ = rig.timed(rig.value_step, K, 0, first=W)
    host_ms = rig.enqueue_s * 1e3 / K
    value_launches = (abi.kernel_launch_count() - launches0) / K
    ts1 = time.time()
    clocks = sampler.stop(ts0, ts1)
    if args.dump_outputs and rank == 0:          # N > 1: rank 0's rows, and the cluster lists every rank holds
        dump_outputs(args.dump_outputs, ctx, n, V)
    if not args.no_parity:
        fchk = W + K
        if fchk % WIN == 0:        # slot 0's recorded constants carry the feedback of the frame before the recording run
            rig.value_step(fchk); fchk += 1
        parity["errors"] += [f"value: {e}" for e in rig.parity_check(fchk, "value")]
        parity["checked"] = True
    dev_ms, e2e_ms, res_ms, sp_ms = rig.max_over_ranks(dev_ms, e2e_sec * 1e3, max(res_wall, res_dev_ms / 1e3) * 1e3,
                                                       max(sp_wall, sp_dev_ms / 1e3) * 1e3)
    ms_per_step = dev_ms / K
    value = total_entities / (ms_per_step * 1e-3)
    e2e_value = total_entities / (e2e_ms / K * 1e-3)

    # ---- pass C: duration of the dominant kernel, CUDA events around it on the launching stream, taken
    # back to back with the timed loop (no host sync between frames, so clocks stay where they were) --------
    ctx.set_profiling(True)
    PF = min(K, 200)
    for i in range(PF):
        rig.value_step(i)
    t_tile, t_expand, t_cluster, nf = ctx.collect_stage_times_ms()
    ctx.set_profiling(False)
    sanity = ctx.download_frame_stats()
    ctx.use_recorded_frame_constants(None)
    tile_ms_avg, expand_ms_avg, cluster_ms_avg = t_tile / nf, t_expand / nf, t_cluster / nf
    visible_pairs_rank = sum(sanity.visible_count[v] for v in range(V))
    # the write-back kernel alone (CUDA events), for the achieved PCIe rate
    wb_ms = None
    if world == 1:
        rig.sinks(True, True)
        rig.e2e_step(1, True)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        torch.cuda.synchronize()
        ev[0].record(stream)
        for _ in range(5):
            ctx.writeback_columns()
        ev[1].record(stream)
        torch.cuda.synchronize()
        wb_ms = ev[0].elapsed_time(ev[1]) / 5
        rig.sinks(False, False)

    lights_rank = len(rig.scene.light_row)
    perr = torch.tensor([len(parity["errors"])], device=dev)
    if world > 1:
        dist.all_reduce(perr)
    parity_ok = bool(parity["checked"]) and int(perr.item()) == 0

    # ---- SURVEY 8(f) rows (N1, N2, N4): what each costs on this workload; outside every timed region above ------------
    next_rows = None
    if world == 1 and not args.no_next_rows:
        next_rows = measure_next_rows(torch, bb, rig, tile_ms_avg, expand_ms_avg, cluster_ms_avg, res_ms / K2, W)

    # ---- N > 1: a short measurement of the other scaling mode, reported beside the primary one -----------------------------
    secondary = None
    if world > 1 and not args.no_secondary:
        other = "weak" if scaling == "strong" else "strong"
        rig.close()
        rig2 = Rig(args, torch, dist, bb, scenes, parallel, other, world, rank, local_rank, dev, stream)
        rig2.ctx.run(bb.STAGE_ALL); rig2.pipe.read_feedback()
        rig2.value_setup()
        K3 = max(100, min(K, 500))
        d_ms, _ = rig2.timed(rig2.value_step, K3, W)
        rig2.sinks(True, True)
        e_dev, e_wall = rig2.timed(lambda f: rig2.e2e_step(f % WIN, True), K3, W)
        rig2.sinks(False, False)
        d_ms, e_ms = rig2.max_over_ranks(d_ms, max(e_wall, e_dev / 1e3) * 1e3)
        tot = (args.trees * PER_TREE + args.lights) * (world if other == "weak" else 1)
        secondary = {"scaling": other, "entities_total": tot, "steps": K3, "value": tot / (d_ms / K3 * 1e-3), "ms_per_step": d_ms / K3,
                     "e2e_value": tot / (e_ms / K3 * 1e-3), "e2e_ms_per_step": e_ms / K3}
        rig = rig2

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak = json.load(open(peaks_path))["hbm_gbs"]; peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        else:
            peak = 6650.0; peak_src = "fallback (B200_PROFILING.md)"
        # DRAM bytes of one launch of the dominant kernel, from the committed `ncu --set full` capture of this workload
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "tile_kernel_traffic.json")
        if os.path.exists(tp) and world == 1:
            tj = json.load(open(tp))
            if tj.get("entities") == n:
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
        algo_bytes = n * ALGO_BYTES_PER_ENTITY + 4 * visible_pairs_rank
        achieved = algo_bytes / (tile_ms_avg * 1e-3) / 1e9
        tile_kernel = {"c": "k_propagate_cull", "s": "k_propagate_cull_scout", "w": "k_tile_warp", "f": "k_propagate_cull_flow",
                       "t": "k_propagate_cull_tma"}.get(os.environ.get("B200VIS_TILE_KERNEL", "l")[:1], "k_propagate_cull_lean")
        cfg_out = dict(cfg)
        line = {
            "metric": METRIC, "value": value, "unit": "entities/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg_out,
            "value_note": "pipelined throughput: frames enqueued back to back, the tail of frame f (list expansion, clusters) overlaps "
                          "the tile pass of frame f+1; the latency of one live frame (feedback loop closed) is what e2e measures",
            "run": {"entities_per_gpu": n, "lights_per_gpu": lights_rank,
                    "sharding": ("contiguous row ranges (whole trees) per GPU; " +
                                 ("cluster x light bit slabs (+ Clusters feedback trailer)" if os.environ.get("B200VIS_EXCHANGE_WHAT", "r")[:1] == "s"
                                  else "light-record blocks (28 B per light), cluster stage on every rank over all lights,") + " exchanged by " +
                                 ("peer stores over NVLink (CUDA IPC) + per-frame stamps" if rig.exchange == "p2p" else "one ncclAllGather"))
                    if world > 1 else "single GPU",
                    "visible_pairs_last_frame": int(visible_pairs), "cluster_indices_last_frame": int(cluster_indices)},
            "clocks": clocks,
            "parity_checked": parity_ok,
            "parity": {"what": "the frame after each timed loop (e2e pass and device-resident pass), every rank, bit-exact vs the CPU oracle: "
                               "GlobalTransform bits, Changed<GlobalTransform>, ViewVisibility, Changed<ViewVisibility>, sorted visible lists, "
                               "cluster offsets/indices/feedback, column write-back mirror and change bits", "errors": parity["errors"]},
            "e2e": {"value": e2e_value, "unit": "entities/s", "h2d_bytes_per_step": int(e2e_h2d), "d2h_bytes_per_step": int(e2e_d2h),
                    "ms_per_step": e2e_ms / K, "device_breakdown": e2e_breakdown, "gt_rows_written_back_per_step": gt_changed_e2e,
                    "pcie": pcie, "writeback_kernel_ms": wb_ms,
                    "writeback_achieved_gbs": (64 * gt_changed_e2e + n + 8 * ((n + 31) // 32)) / (wb_ms * 1e-3) / 1e9 if wb_ms else None,
                    "note": "one b200vis_step per frame: root Transforms from pinned host memory, per-view constants on the host, all kernels, "
                            "the GPU writes stats + sorted visible lists + cluster lists + every changed GlobalTransform (64-byte Affine3A) + "
                            "ViewVisibility bytes + both change-bit sets into host memory; one stream sync"},
            "e2e_resident": {"value": total_entities / (res_ms / K2 * 1e-3), "unit": "entities/s", "ms_per_step": res_ms / K2, "steps": K2,
                             "d2h_bytes_per_step": int(res_d2h),
                             "note": "GlobalTransform / ViewVisibility columns stay on the device (round 1's e2e)"},
            "e2e_sparse": {"value": total_entities / (sp_ms / K2 * 1e-3), "unit": "entities/s", "ms_per_step": sp_ms / K2, "steps": K2,
                           "d2h_bytes_per_step": int(sp_d2h), "gt_rows_written_back_per_step": sp_changed,
                           "note": "the reference bench's own mutation pattern: 8 roots move per frame (propagate.rs:115-128), full write-back"},
            "gpu_launches": int(round(value_launches * K)), "gpu_launches_per_step": value_launches, "gpu_launches_per_e2e_step": e2e_launches,
            "host_enqueue_ms_per_step": host_ms,
            "roofline": {"bound": "hbm", "kernel": tile_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel_ms": tile_ms_avg, "expand_ms": expand_ms_avg, "cluster_ms": cluster_ms_avg,
                         "gt_changed_rows_last_frame": int(sanity.gt_changed_count),
                         "algorithmic_bytes_per_entity": ALGO_BYTES_PER_ENTITY, "note": EXTRA_BYTES_NOTE},
        }
        if secondary is not None:
            line["secondary_scaling"] = secondary
        if next_rows is not None:
            line["next_rows"] = next_rows
        if not args.no_cpu_baseline:
            cpu_scene = scenes.forest(args.trees, LEVELS, args.lights)
            arm = CpuArm(cpu_scene)
            times = arm.run(args.cpu_frames, 3)
            line["cpu_baseline"] = cpu_summary(times, cpu_scene.n, arm.threads,
                                               f"{args.cpu_frames} frames of the same {cpu_scene.n}-entity workload after 3 warm-up frames",
                                               arm.calibration)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    rig.close()


if __name__ == "__main__":
    main()
