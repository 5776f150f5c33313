"""Cost of updating a resident mesh on the device (GpuContext.update_mesh) next to rebuilding the host Scene and
uploading it again, and whether updates stall frames in flight; one JSON line per workload.

   python tools/bench_update.py [--reps 20] [--warmup 3] [--out FILE]

Workloads:
  update_<mesh>  update_mesh of TorusKnot, unitychan (21 760 triangles with the stand-ins) and a grid of TorusKnot copies
                 of about 1 M triangles (tools/make_c5.py, copies = 1 M / the knot's triangles), new points from a per-vertex wobble made by torch on the device.
                 build_ms: device time of the call on its stream (CUDA events around it: input check, tree build,
                 shading records, bounds, publish); call_ms: host wall time of the call (it returns once the build is
                 complete).  rebuild_upload_ms: host wall time of Scene(spec) from the OBJ plus upload_scene.
  frames_4k      PATH frames of unitychan at 3840 x 2160 (MaxBounceTimes 10, one un-jittered ray per pixel) round-robin
                 on four frame slots, with and without one on-device deformation plus update_mesh per frame on
                 torch's stream; frames_per_s over --reps frames after --warmup.
Medians of --reps after --warmup.  The device name and power limit are read with nvidia-smi (query only).
"""
import argparse
import json
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
import make_c5  # noqa: E402
from bench_queries import device_info  # noqa: E402


def wobble(torch, p0, t):
    return (p0 + 0.02 * torch.sin(3.0 * p0[:, [1, 2, 0]] + t)).contiguous()


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, power = device_info()
    scratch = tempfile.TemporaryDirectory(prefix="rtb200_bu_")
    data = os.path.join(ROOT, "assets", "_ref", "Data")
    stand_ins = not os.path.isdir(data)
    if stand_ins:
        import standin_data
        data = standin_data.write(os.path.join(scratch.name, "Data"))
    assets = "generated stand-ins of the reference's meshes (tests/standin_data.py)" if stand_ins else "reference meshes"
    grid = os.path.join(scratch.name, "grid.obj")
    knot_tris = rt.Scene([("mesh", os.path.join(data, "TorusKnot.obj"), None)]).mesh_counts(0)[3]
    make_c5.main(os.path.join(data, "TorusKnot.obj"), grid, max(1, round(1_000_000 / knot_tris)))      # ~1 M triangles
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    lines = []

    def emit(d):
        d.update(device=name, power_limit=power, assets=assets, reps=args.reps, warmup=args.warmup)
        line = json.dumps(d)
        print(line, flush=True)
        lines.append(line)

    for label, path in (("torusknot", os.path.join(data, "TorusKnot.obj")), ("unitychan", os.path.join(data, "unitychan.obj")),
                        ("grid", grid)):
        spec = [("mesh", path, ("diffuse", (1, 1, 1)))]
        sc = rt.Scene(spec)
        dump = sc.mesh_dump(0)
        ctx = rt.GpuContext(0)
        ctx.upload_scene(sc)
        p0 = torch.from_numpy(dump["points"]).to(dev)
        idx = torch.from_numpy(dump["pidx"].reshape(-1, 3)).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        build, call = [], []
        for i in range(args.warmup + args.reps):
            pts = wobble(torch, p0, float(i))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record(stream)
            ctx.update_mesh(0, pts, idx)
            e1.record(stream)
            t1 = time.perf_counter()
            torch.cuda.synchronize()
            if i >= args.warmup:
                build.append(e0.elapsed_time(e1)); call.append((t1 - t0) * 1e3)
        ctx.close()
        up = []
        for i in range(args.warmup + min(args.reps, 5)):
            ctx = rt.GpuContext(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s2 = rt.Scene(spec)
            ctx.upload_scene(s2)
            t1 = time.perf_counter()
            ctx.close()
            if i >= args.warmup:
                up.append((t1 - t0) * 1e3)
        emit(dict(workload=f"update_{label}", triangles=int(len(dump["pidx"]) // 3), points=int(len(dump["points"])),
                  build_ms=float(np.median(build)), call_ms=float(np.median(call)),
                  rebuild_upload_ms=float(np.median(up))))

    # frames in flight with and without an update per frame
    sc = rt.Scene(scenes.c3_unitychan(data))
    sc.set_unit_vectors(seed=0)
    dump = sc.mesh_dump(0)
    W, H = 3840, 2160
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, pass_count=1, antialias=0, seed=1)
    res = {}
    for with_updates in (False, True):
        ctx = rt.GpuContext(0)
        ctx.upload_scene(sc)
        p0 = torch.from_numpy(dump["points"]).to(dev)
        idx = torch.from_numpy(dump["pidx"].reshape(-1, 3)).to(dev)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.reset_accum(W, H)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.synchronize()
        t0 = None
        for i in range(args.warmup + args.reps):
            if i == args.warmup:
                for s in range(4):
                    ctx.set_frame_slot(s)
                    ctx.synchronize()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            if with_updates:
                ctx.update_mesh(0, wobble(torch, p0, float(i)), idx)
            ctx.set_frame_slot(i % 4)
            p.pass_begin = i
            ctx.render_tile(p)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.synchronize()
        torch.cuda.synchronize()
        res[with_updates] = args.reps / (time.perf_counter() - t0)
        ctx.close()
    emit(dict(workload="frames_4k", width=W, height=H, slots=4, frames_per_s_no_updates=res[False],
              frames_per_s_with_updates=res[True]))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
