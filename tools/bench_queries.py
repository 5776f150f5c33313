"""Throughput of ray queries on device memory (GpuContext.query_rays), one JSON line per batch.

   python tools/bench_queries.py [--reps 20] [--warmup 3]

Workloads (unitychan, tests/scenes.py c3_unitychan, unless named otherwise):
  pinhole_blocks   the reference's camera for a 3840 x 2160 frame, un-jittered, in the 8x4-pixel block order of the
                   render's work list (round-0 packets of 32 coherent rays)
  pinhole_shuffled the same rays in random order (packets are given up and walked lane by lane)
  bounce           8 M bounce-like rays from the primary hit points (origin off the surface, into the hemisphere)
  default_scene    the pinhole batch against RayTracerProgram::SetupScene (spheres, capsule, ground plane, unitychan)
Each batch is timed as a nearest-hit and as an occlusion query, culled traversal, with CUDA events on the query's
stream (median of --reps after --warmup), and counted once in exact mode for the reference's slab / triangle tests.
Next to it: the test hook rt_gpu_trace_rays on the same rays (host arrays in and out: its wall time INCLUDES the
host-device copies and allocations), and for the pinhole batch render_tile(RT_MODE_PRIMARY, antialias=0) of the same
4K frame, which does the same work through the camera generator.  unitychan's geometry (~2 MB of nodes and
triangles) stays resident in the 126 MB L2, so these are L2-bound walk rates, not HBM-bound ones.
The device name and power limit are read with nvidia-smi (query only) and go into every line.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import raytracerwin_b200 as rt  # noqa: E402
import scenes  # noqa: E402
from test_ray_queries import bounce_rays, pinhole_rays  # noqa: E402


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             check=True, capture_output=True, text=True).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:          # the numbers are still printed, without the card's identity
        return f"unknown ({e})", "unknown"


def median_ms(fn, stream, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        fn()
        t1.record(stream)
        t1.synchronize()
        times.append(t0.elapsed_time(t1))
    return float(np.median(times))


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--hook-reps", type=int, default=3)
    args = ap.parse_args()
    name, power = device_info()
    data = os.path.join(ROOT, "assets", "_ref", "Data")
    scratch = None
    if not os.path.isdir(data):
        import standin_data
        scratch = tempfile.TemporaryDirectory(prefix="rtb200_bq_")
        data = standin_data.write(os.path.join(scratch.name, "Data"))
    assets = "reference meshes" if scratch is None else "generated stand-ins of the reference's meshes (tests/standin_data.py)"
    W, H = 3840, 2160
    ctx = rt.GpuContext(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    blocks = pinhole_rays(W, H, True)
    shuffled = blocks[np.random.default_rng(1).permutation(len(blocks))]
    uc = rt.Scene(scenes.c3_unitychan(data))
    ctx.upload_scene(uc)
    primary = ctx.trace_rays(blocks, rt.RT_TRAVERSE_CULLED)
    bounce = bounce_rays(primary[2], 8_000_000, 2)
    default = rt.Scene(scenes.default_scene(data))
    for scene_name, sc, workload, rays in (("unitychan", uc, "pinhole_blocks", blocks), ("unitychan", uc, "pinhole_shuffled", shuffled),
                                           ("unitychan", uc, "bounce", bounce), ("default_scene", default, "pinhole_blocks", blocks)):
        ctx.upload_scene(sc)
        d = torch.from_numpy(rays).to(dev)
        n = len(rays)
        for any_hit in (False, True):
            ms = median_ms(lambda: ctx.query_rays(d, any_hit=any_hit), stream, args.reps, args.warmup)
            stats = {}
            for tr, key in ((rt.RT_TRAVERSE_CULLED, "culled"), (rt.RT_TRAVERSE_EXACT, "exact")):
                ctx.synchronize()
                ctx.reset_counters()
                ctx.synchronize()
                ctx.query_rays(d, any_hit=any_hit, traverse=tr)
                torch.cuda.synchronize()
                stats[key] = ctx.counters()
            c = stats["culled"]
            line = dict(device=name, power_limit=power, assets=assets, scene=scene_name, workload=workload, n=n,
                        kind="any" if any_hit else "nearest", traverse="culled", query_ms=round(ms, 3),
                        grays_per_s=round(n / ms / 1e6, 3), g_mesh_walks_per_s=round(c["mesh_walks"] / ms / 1e6, 3),
                        node_visits_per_ray=round(c["node_visits"] / n, 2),
                        exact_node_tests_per_ray=round(stats["exact"]["node_tests"] / n, 2))
            if not any_hit:
                hook = []
                for _ in range(args.hook_reps):
                    t = time.perf_counter()
                    ctx.trace_rays(rays, rt.RT_TRAVERSE_CULLED)
                    hook.append((time.perf_counter() - t) * 1e3)
                line["hook_wall_ms_incl_copies"] = round(float(np.median(hook)), 3)
            if workload == "pinhole_blocks" and not any_hit:
                p = rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, antialias=0, traverse=rt.RT_TRAVERSE_CULLED)
                ctx.reset_accum(W, H)
                rend = []
                for i in range(args.warmup + args.reps):
                    ctx.render_tile(p)
                    if i >= args.warmup:
                        rend.append(ctx.last_render_ms())
                line["render_primary_4k_ms"] = round(float(np.median(rend)), 3)
            print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
