"""Throughput of radiance queries on device memory (GpuContext.radiance_rays) next to render_tile of the same frame,
one JSON line per workload.

   python tools/bench_radiance.py [--reps 20] [--warmup 3] [--out FILE]

Workloads:
  path_4k     unitychan (tests/scenes.py c3_unitychan, the reference's unit-vector table), RT_MODE_PATH with
              MaxBounceTimes 10, the reference's camera for a 3840 x 2160 frame, one un-jittered ray per pixel, ray i
              drawing from the stream of its pixel.  The rays go in three orders: the 8x4-pixel blocks of the render's work
              list (round-0 packets of 32 coherent rays), row order, and shuffled (packets are given up and walked lane by
              lane).  Every order computes the same paths; only their grouping differs.  Next to it:
              render_tile(RT_MODE_PATH, antialias=0, pass_count=1) of the same frame, which makes its camera rays itself.
  whitted_c1  TorusKnot (c1_torusknot), RT_MODE_WHITTED, 640 x 480, block order, against render_tile(RT_MODE_WHITTED).
Queries are timed with CUDA events on the query's stream, renders with rt_gpu_last_render_ms (CUDA events on the
context's stream); median of --reps after --warmup.  A query reads 28 B of ray and 4 B of stream id and writes 16 B of
radiance per ray that the render's generator does not move, and the render folds four sky samples of a pixel in its
generate kernel (not used here: one ray per pixel).  The device name and power limit are read with nvidia-smi (query
only) and go into every line, with the meshes used (the reference's or the generated stand-ins).
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracerwin_b200 as rt  # noqa: E402
import scenes  # noqa: E402
from bench_queries import device_info, median_ms  # noqa: E402
from test_ray_queries import pinhole_rays  # noqa: E402


def pixel_ids(W, H, block_order):
    """the pixel of each ray of pinhole_rays(W, H, block_order)"""
    if not block_order:
        return np.arange(W * H, dtype=np.int32)
    lane = np.arange(32)
    bx, by = np.meshgrid(np.arange(W // 8), np.arange(H // 4))
    x = (bx.reshape(-1, 1) * 8 + (lane & 7)).reshape(-1)
    y = (by.reshape(-1, 1) * 4 + (lane >> 3)).reshape(-1)
    return (y * W + x).astype(np.int32)


def render_ms(ctx, p, reps, warmup):
    ctx.reset_accum(p.width, p.height)
    times = []
    for i in range(warmup + reps):
        ctx.render_tile(p)
        if i >= warmup:
            times.append(ctx.last_render_ms())
    return float(np.median(times))


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, power = device_info()
    data = os.path.join(ROOT, "assets", "_ref", "Data")
    scratch = None
    if not os.path.isdir(data):
        import standin_data
        scratch = tempfile.TemporaryDirectory(prefix="rtb200_br_")
        data = standin_data.write(os.path.join(scratch.name, "Data"))
    assets = "reference meshes" if scratch is None else "generated stand-ins of the reference's meshes (tests/standin_data.py)"
    ctx = rt.GpuContext(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    lines = []

    def emit(line):
        line = dict(device=name, power_limit=power, assets=assets, **line)
        lines.append(line)
        print(json.dumps(line), flush=True)

    for workload, scene, spec, mode, W, H, bounce in (
            ("path_4k", "unitychan", scenes.c3_unitychan(data), rt.RT_MODE_PATH, 3840, 2160, 10),
            ("whitted_c1", "TorusKnot", scenes.c1_torusknot(data), rt.RT_MODE_WHITTED, 640, 480, 10)):
        sc = rt.Scene(spec)
        sc.set_unit_vectors(seed=0, count=0)
        ctx.upload_scene(sc)
        p = rt.make_params(W, H, mode=mode, max_bounce=bounce, antialias=0, pass_count=1, seed=1)
        ms_render = render_ms(ctx, p, args.reps, args.warmup)
        ctx.synchronize()
        ctx.reset_counters()
        ctx.render_tile(p)
        ctx.synchronize()
        rc = ctx.counters()
        blocks = pinhole_rays(W, H, True)
        orders = [("blocks", blocks, pixel_ids(W, H, True))]
        if workload == "path_4k":
            perm = np.random.default_rng(1).permutation(len(blocks))
            orders += [("rows", pinhole_rays(W, H, False), pixel_ids(W, H, False)),
                       ("shuffled", blocks[perm], pixel_ids(W, H, True)[perm])]
        for order, rays, ids in orders:
            d = torch.from_numpy(rays).to(dev)
            s = torch.from_numpy(ids).to(dev)
            out = torch.empty((len(rays), 4), dtype=torch.float32, device=dev)
            n = len(rays)
            ms = median_ms(lambda: ctx.radiance_rays(d, mode=mode, max_bounce=bounce, seed=1, rng_stream=s, out=out),
                           stream, args.reps, args.warmup)
            torch.cuda.synchronize()
            ctx.synchronize()
            ctx.reset_counters()
            ctx.synchronize()
            ctx.radiance_rays(d, mode=mode, max_bounce=bounce, seed=1, rng_stream=s, out=out)
            torch.cuda.synchronize()
            c = ctx.counters()
            emit(dict(workload=workload, scene=scene,
                      mode={rt.RT_MODE_PATH: "path", rt.RT_MODE_WHITTED: "whitted"}[mode], max_bounce=bounce,
                      width=W, height=H, order=order, n=n, traverse="culled", query_ms=round(ms, 3),
                      render_ms=round(ms_render, 3), query_over_render=round(ms / ms_render, 3),
                      grays_per_s=round(c["rays"] / ms / 1e6, 3), render_grays_per_s=round(rc["rays"] / ms_render / 1e6, 3),
                      rays_per_query=round(c["rays"] / n, 3), rays_per_render_camera_ray=round(rc["rays"] / rc["camera_rays"], 3),
                      shadow_rays=c["shadow_rays"]))
    ctx.close()
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
