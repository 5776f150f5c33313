"""Cost of a camera per render call (GpuContext.render_tile(params, camera), rt_gpu_render_view); one JSON line per
workload.

   python tools/bench_camera.py [--reps 20] [--warmup 3] [--out FILE]

Workloads (unitychan, tests/scenes.py c3_unitychan):
  overhead_c3_4k  the C3/C4 frame: 3840 x 2160, PATH, MaxBounceTimes 10, 16 camera rays/pixel (4 passes x 4 jittered)
                  as render_tile, as render_view with the identity camera of the uploaded view, and as render_view with
                  that camera turned by 1e-3 rad about y (nearly the same work, through the view variant of the generate
                  kernel).  Device time per frame (the call's own events, rt_gpu_last_render_ms), median of --reps, the
                  three variants alternating within each rep.
  framed_4k       the same frame from close look_at cameras (unitychan's box taller than the frame), next to the default view:
                  Grays/s (rays / device time), mesh walks and node visits (culled traversal) per ray.
  orbit_4k        the 4-slot 4K PATH frame loop of tools/bench_update.py (one un-jittered ray per pixel, MaxBounceTimes
                  10), frames/s three ways: one fixed orbit camera, a new orbit camera every frame through render_view,
                  and the orbit's eye through upload_scene every frame (a new scene eye; the basis cannot turn that way).
The device name and power limit are read with nvidia-smi (query only) and go into every line.
"""
import argparse
import json
import math
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracerwin_b200 as rt  # noqa: E402
import scenes  # noqa: E402
from bench_queries import device_info  # noqa: E402


def mesh_box(sc):
    s = sc.desc.contents.shapes[0]
    lo, hi = np.array(list(s.bounds_min), np.float64), np.array(list(s.bounds_max), np.float64)
    return (lo + hi) / 2, (hi - lo) / 2


def framing(center, half, yaw):
    """look_at from direction `yaw` about y, close enough that the mesh's box is taller than the frame (tan of the
    vertical half-angle is 0.25 / 0.5 at dir_z = -0.5; the figure covers a small part of its box)"""
    dist = 0.35 * half[1] / 0.5 + max(half[0], half[2])
    eye = center + dist * np.array([math.sin(yaw), 0.0, math.cos(yaw)])
    return rt.look_at(eye, center)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, power = device_info()
    scratch = tempfile.TemporaryDirectory(prefix="rtb200_bc_")
    data = os.path.join(ROOT, "assets", "_ref", "Data")
    stand_ins = not os.path.isdir(data)
    if stand_ins:
        import standin_data
        data = standin_data.write(os.path.join(scratch.name, "Data"))
    assets = "generated stand-ins of the reference's meshes (tests/standin_data.py)" if stand_ins else "reference meshes"
    lines = []

    def emit(d):
        d.update(device=name, power_limit=power, assets=assets, reps=args.reps, warmup=args.warmup)
        line = json.dumps(d)
        print(line, flush=True)
        lines.append(line)

    sc = rt.Scene(scenes.c3_unitychan(data))
    sc.set_unit_vectors(seed=0)
    d = sc.desc.contents
    center, half = mesh_box(sc)
    W, H = 3840, 2160

    # ---- overhead: render_tile, the identity camera, a camera turned by 1e-3 rad ---------------------------------
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, pass_count=4, seed=1)
    eye = list(d.eye)
    ident = rt.camera(eye, (1, 0, 0), (0, 1, 0), (0, 0, 1), d.dir_z, d.ray_distance)
    a = 1e-3
    turned = rt.camera(eye, (math.cos(a), 0, -math.sin(a)), (0, 1, 0), (math.sin(a), 0, math.cos(a)), d.dir_z, d.ray_distance)
    variants = (("render_tile", None), ("identity", ident), ("turned_1e-3", turned))
    times = {k: [] for k, _ in variants}
    rays = {}
    for i in range(args.warmup + args.reps):
        for k, cam in variants:
            ctx.reset_accum(W, H)
            ctx.reset_counters()
            ctx.render_tile(p, cam)
            ctx.synchronize()
            if i >= args.warmup:
                times[k].append(ctx.last_render_ms())
                rays[k] = ctx.counters()["rays"]
    emit(dict(workload="overhead_c3_4k", width=W, height=H, camera_rays_per_pixel=16, max_bounce=10,
              **{f"ms_{k}": float(np.median(v)) for k, v in times.items()},
              **{f"ms_spread_{k}": [float(np.min(v)), float(np.max(v))] for k, v in times.items()},
              **{f"rays_{k}": int(v) for k, v in rays.items()}))

    # ---- a framed view against the default view ------------------------------------------------------------------
    views = (("default_view", None), ("framed_front", framing(center, half, 0.0)), ("framed_side", framing(center, half, 1.2)))
    for k, cam in views:
        ms = []
        for i in range(args.warmup + args.reps):
            ctx.reset_accum(W, H)
            ctx.reset_counters()
            ctx.render_tile(p, cam)
            ctx.synchronize()
            if i >= args.warmup:
                ms.append(ctx.last_render_ms())
        c = ctx.counters()
        # the share of camera rays that see only sky, from one un-jittered PRIMARY pass
        ctx.reset_accum(W, H)
        ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, antialias=0, seed=1), cam)
        ctx.synchronize()
        sky = float((ctx.readback(rt.RT_READ_PRIMARY_IDS_I32X2, W, H)[..., 0] < 0).mean())
        t = float(np.median(ms))
        emit(dict(workload="framed_4k", view=k, width=W, height=H, camera_rays_per_pixel=16, max_bounce=10,
                  ms=t, grays_per_s=c["rays"] / t / 1e6, rays=c["rays"], mesh_walks_per_ray=c["mesh_walks"] / c["rays"],
                  node_visits_per_ray=c["node_visits"] / c["rays"], sky_share=sky,
                  eye=None if cam is None else [float(x) for x in cam.eye]))
    ctx.close()

    # ---- orbit loop on four frame slots --------------------------------------------------------------------------
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, pass_count=1, antialias=0, seed=1)
    n = args.warmup + args.reps
    orbit = [framing(center, half, 2 * math.pi * i / max(n, 1)) for i in range(n)]
    res = {}
    for how in ("fixed", "render_view", "upload_scene"):
        ctx = rt.GpuContext(0)
        ctx.upload_scene(sc)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.reset_accum(W, H)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.synchronize()
        t0 = None
        for i in range(n):
            if i == args.warmup:
                for s in range(4):
                    ctx.set_frame_slot(s)
                    ctx.synchronize()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            cam = None
            if how == "fixed":
                cam = orbit[0]
            elif how == "render_view":
                cam = orbit[i]
            else:
                for k in range(3):
                    d.eye[k] = orbit[i].eye[k]
                ctx.upload_scene(sc)
            ctx.set_frame_slot(i % 4)
            p.pass_begin = i
            ctx.render_tile(p, cam)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.synchronize()
        torch.cuda.synchronize()
        res[how] = args.reps / (time.perf_counter() - t0)
        ctx.close()
    emit(dict(workload="orbit_4k", width=W, height=H, slots=4, camera_rays_per_pixel=1, max_bounce=10,
              frames_per_s_fixed_camera=res["fixed"], frames_per_s_render_view_orbit=res["render_view"],
              frames_per_s_upload_scene_orbit=res["upload_scene"]))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
