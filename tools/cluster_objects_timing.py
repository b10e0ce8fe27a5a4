"""Cost of clustering rect lights, light probes and clustered decals (b200vis_set_clusterable_objects) on the bench workload.

Config #3 (3922 trees x 255 nodes + 256 point lights, 4 views) with 64 rect lights, 128 probes and 256 decals appended as
children of moving roots.  Two contexts on the same scene: one clusters the point lights only, the other the point lights
and the objects (the object rows are propagated and culled in both).  For each: the pipelined device-resident step time
(upload + run(ALL), CUDA events over the loop, as bench.py's `value`) and the cluster stage time from
b200vis_collect_stage_times_ms.  The two contexts alternate over several rounds so that the spread is visible.  Prints the
card's name and power limit first.  Needs a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bevy_b200 as bb  # noqa: E402
from bevy_b200 import scenes  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


class Arm:
    def __init__(self, sc, objects, stream):
        self.name = "with objects" if objects else "point lights only"
        self.pipe = bb.VisibilityPipeline(sc, max_lights=len(sc.light_row) + len(sc.obj_kind))
        self.ctx = self.pipe.ctx
        self.ctx.set_stream(stream.cuda_stream)
        if objects:
            self.ctx.set_clusterable_objects(sc.obj_kind, sc.obj_row, sc.obj_range, sc.obj_layers)
        for _ in range(3):                               # settle the cluster grid through the feedback
            self.pipe.update_views(); self.pipe.run_frame(); self.pipe.read_feedback()
        self.pipe.update_views_fast()
        self.ctx.use_recorded_frame_constants(self.ctx.record_frame_constants())
        self.stats = self.ctx.download_frame_stats()


def time_arm(arm, stream, rows_d, frames, steps, warmup):
    ctx, n = arm.ctx, rows_d.numel()

    def one(i):
        ctx.upload_transforms_scattered_raw(n, rows_d.data_ptr(), frames[i % len(frames)].data_ptr())
        ctx.run(bb.STAGE_ALL)
    for i in range(warmup):
        one(i)
    ctx.join(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        one(i)
    ctx.join(); e1.record(stream); torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    ctx.set_profiling(True)                              # stage times in a separate pass: the events serialise a little
    for i in range(min(steps, 256)):
        one(i)
    tile_ms, expand_ms, cluster_ms, nf = ctx.collect_stage_times_ms()
    ctx.set_profiling(False)
    return step_ms, tile_ms / max(nf, 1), cluster_ms / max(nf, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--rect", type=int, default=64)
    ap.add_argument("--probes", type=int, default=128)
    ap.add_argument("--decals", type=int, default=256)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    print("card:", card())
    sc = scenes.add_clusterable_objects(scenes.forest(3922, 8, 256), a.rect, a.probes, a.decals)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    arms = [Arm(sc, False, stream), Arm(sc, True, stream)]
    frames = [torch.from_numpy(np.ascontiguousarray(scenes.mutate_roots(sc, f + 1)[1], np.float32)).cuda() for f in range(8)]
    rows_d = torch.from_numpy(sc.roots.astype(np.int32)).cuda()
    ordinals = [len(sc.light_row), len(sc.light_row) + len(sc.obj_kind)]
    for arm, n_ord in zip(arms, ordinals):
        print(f"{arm.name}: {n_ord} ordinals, cluster index counts per view {list(arm.stats.cluster_index_count)[:len(sc.cameras)]}")
    results = {arm.name: [] for arm in arms}
    for r in range(a.rounds):
        for arm in arms:
            step_ms, tile_ms, cluster_ms = time_arm(arm, stream, rows_d, frames, a.steps, a.warmup)
            results[arm.name].append(dict(step_us=1e3 * step_ms, tile_us=1e3 * tile_ms, cluster_us=1e3 * cluster_ms))
            print(f"round {r} {arm.name:18s} step {1e3 * step_ms:7.2f} us  tile {1e3 * tile_ms:7.2f} us  cluster {1e3 * cluster_ms:6.2f} us")
    print(json.dumps({"card": card(), "rows": sc.n, "objects": dict(rect=a.rect, probes=a.probes, decals=a.decals),
                      "results": results}))
    for arm in arms:
        arm.pipe.close()


if __name__ == "__main__":
    main()
