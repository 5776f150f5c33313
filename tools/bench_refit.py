"""Cost of refitting a resident mesh on the device (GpuContext.refit_mesh) next to rebuilding its tree
(GpuContext.update_mesh), in frames in flight, and in walk time afterwards; one JSON line per workload.

   python tools/bench_refit.py [--reps 20] [--warmup 3] [--out FILE]

Workloads:
  refit_<mesh>   refit_mesh of TorusKnot, unitychan (21 760 triangles with the stand-ins) and tools/bench_update.py's grid
                 of TorusKnot copies (about 1 M triangles), new points from bench_update's per-vertex wobble made by
                 torch on the device.  refit_ms: device time of the call on its stream (CUDA events around it);
                 call_ms: host wall time of the call (it returns at once); update_ms: update_mesh's device time on the
                 same points in the same run.
  frames_4k      bench_update's loop: PATH frames of unitychan at 3840 x 2160 (MaxBounceTimes 10, one un-jittered ray
                 per pixel) round-robin on four frame slots, with no geometry change, with a wobble plus update_mesh per
                 frame, and with a wobble plus refit_mesh per frame; frames_per_s over --reps frames after --warmup.
  refit_quality  render_tile ms of that 4K frame (one slot, the context's own timing) after update_mesh and after
                 refit_mesh of the same deformed points: the wobble, and a rigid rotation by 45 degrees about x then
                 45 degrees about y (boxes fitted around the turned subtrees of the uploaded tree are no longer tight:
                 a rotation by 90 degrees would map boxes to boxes).  undeformed_ms: the uploaded geometry.
Medians of --reps after --warmup.  The device name and power limit are read with nvidia-smi (query only).
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
import make_c5  # noqa: E402
from bench_queries import device_info  # noqa: E402
from bench_update import wobble  # noqa: E402


def rotation(torch, p0, dev):
    a = math.pi / 4
    rx = torch.tensor([[1, 0, 0], [0, math.cos(a), -math.sin(a)], [0, math.sin(a), math.cos(a)]], dtype=torch.float32)
    ry = torch.tensor([[math.cos(a), 0, math.sin(a)], [0, 1, 0], [-math.sin(a), 0, math.cos(a)]], dtype=torch.float32)
    return (p0 @ (ry @ rx).T.to(dev)).contiguous()


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, power = device_info()
    scratch = tempfile.TemporaryDirectory(prefix="rtb200_br_")
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
        sc = rt.Scene([("mesh", path, ("diffuse", (1, 1, 1)))])
        dump = sc.mesh_dump(0)
        ctx = rt.GpuContext(0)
        ctx.upload_scene(sc)
        p0 = torch.from_numpy(dump["points"]).to(dev)
        idx = torch.from_numpy(dump["pidx"].reshape(-1, 3)).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = {"refit": [], "call": [], "update": []}
        for op in ("refit", "update"):
            for i in range(args.warmup + args.reps):
                pts = wobble(torch, p0, float(i))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e0.record(stream)
                if op == "refit":
                    status = ctx.refit_mesh(0, pts, idx)
                else:
                    ctx.update_mesh(0, pts, idx)
                e1.record(stream)
                t1 = time.perf_counter()
                torch.cuda.synchronize()
                if op == "refit" and status.item() != 0:
                    raise RuntimeError(f"refit_mesh status {status.item()}")
                if i >= args.warmup:
                    times[op].append(e0.elapsed_time(e1))
                    if op == "refit":
                        times["call"].append((t1 - t0) * 1e3)
        ctx.close()
        T = int(len(dump["pidx"]) // 3)
        emit(dict(workload=f"refit_{label}", triangles=T, points=int(len(dump["points"])),
                  refit_ms=float(np.median(times["refit"])), call_ms=float(np.median(times["call"])),
                  update_ms=float(np.median(times["update"]))))

    # frames in flight with no change, an update per frame, a refit per frame
    sc = rt.Scene(scenes.c3_unitychan(data))
    sc.set_unit_vectors(seed=0)
    dump = sc.mesh_dump(0)
    W, H = 3840, 2160
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, pass_count=1, antialias=0, seed=1)
    res = {}
    for op in ("none", "update", "refit"):
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
            if op == "update":
                ctx.update_mesh(0, wobble(torch, p0, float(i)), idx)
            elif op == "refit":
                ctx.refit_mesh(0, wobble(torch, p0, float(i)), idx)
            ctx.set_frame_slot(i % 4)
            p.pass_begin = i
            ctx.render_tile(p)
        for s in range(4):
            ctx.set_frame_slot(s)
            ctx.synchronize()
        torch.cuda.synchronize()
        res[op] = args.reps / (time.perf_counter() - t0)
        ctx.close()
    emit(dict(workload="frames_4k", width=W, height=H, slots=4, frames_per_s_no_updates=res["none"],
              frames_per_s_with_updates=res["update"], frames_per_s_with_refits=res["refit"]))

    # walk time after a refit against a rebuild of the same points
    def frame_ms(ctx):
        ms = []
        for i in range(args.warmup + args.reps):
            ctx.reset_accum(W, H)
            p.pass_begin = i
            ctx.render_tile(p)
            ctx.synchronize()
            if i >= args.warmup:
                ms.append(ctx.last_render_ms())
        return float(np.median(ms))

    p0 = torch.from_numpy(dump["points"]).to(dev)
    idx = torch.from_numpy(dump["pidx"].reshape(-1, 3)).to(dev)
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)
    undeformed = frame_ms(ctx)
    ctx.close()
    for kind, pts in (("wobble", wobble(torch, p0, 1.0)), ("rotate45", rotation(torch, p0, dev))):
        out = {}
        for op in ("update", "refit"):
            ctx = rt.GpuContext(0)
            ctx.upload_scene(sc)
            if op == "update":
                ctx.update_mesh(0, pts, idx)
            else:
                ctx.refit_mesh(0, pts, idx)
            torch.cuda.synchronize()
            out[op] = frame_ms(ctx)
            ctx.close()
        emit(dict(workload="refit_quality", deformation=kind, width=W, height=H, undeformed_ms=undeformed,
                  after_update_ms=out["update"], after_refit_ms=out["refit"]))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
