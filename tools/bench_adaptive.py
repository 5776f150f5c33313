"""Cost and gain of adaptive sampling (rt_gpu_track_moments, rt_gpu_select_pixels, rt_gpu_render_masked); one JSON
line per workload.

   python tools/bench_adaptive.py [--reps 10] [--warmup 3] [--ref-passes 256] [--out FILE]

Workloads (unitychan, tests/scenes.py c3_unitychan):
  overhead_c3_4k      the C3/C4 frame: 3840 x 2160, PATH, MaxBounceTimes 10, 4 passes x 4 jittered rays, three ways:
                      render_tile, render_tile with moments tracked, and render_tile with an all-ones device mask
                      (rt_gpu_render_masked: compaction, list generate, list fold).  Device time per frame (the call's
                      own events, rt_gpu_last_render_ms), median of --reps, the three variants alternating in each rep.
  convergence_1080p   the close front look_at view of tools/bench_camera.py (framing(yaw = 0)) at 1920 x 1080, PATH,
                      MaxBounceTimes 10, antialiased.  Reference: the mean of --ref-passes uniform passes of other pass
                      indices.  Uniform: passes [0, N) for N = 4, 8, ..., 64.  Adaptive: GpuContext.render_adaptive's
                      loop (min 4, max 64, 4 passes per round) at several tolerances.  For each: device time (the
                      render calls' rt_gpu_last_render_ms, summed; the selection kernel is not in it), wall time of the
                      whole loop (host reads of each round's count included), camera rays, and RMSE of the linear mean
                      colour against the reference.  Each adaptive line also gives the uniform run's camera rays and
                      device time at the same RMSE (log-log interpolation between uniform points) and the ratios.
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
from bench_camera import framing, mesh_box  # noqa: E402
from bench_queries import device_info  # noqa: E402


def mean_image(ctx, W, H):
    a = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    return a[..., :3].astype(np.float64) / np.maximum(a[..., 3:4], 1)


def rmse(img, ref):
    return float(np.sqrt(np.mean((img - ref) ** 2)))


def interp_loglog(x, xs, ys):
    """y at x on the piecewise log-log line through (xs, ys), xs decreasing in y; None outside the points"""
    lx, lxs, lys = math.log(x), np.log(xs), np.log(ys)
    order = np.argsort(lxs)
    lxs, lys = lxs[order], lys[order]
    if lx < lxs[0] or lx > lxs[-1]:
        return None
    return float(np.exp(np.interp(lx, lxs, lys)))


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--ref-passes", type=int, default=256)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, power = device_info()
    scratch = tempfile.TemporaryDirectory(prefix="rtb200_ba_")
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
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)

    # ---- overhead: render_tile, with moments tracked, with an all-ones mask --------------------------------------
    W, H = 3840, 2160
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, pass_count=4, seed=1)
    ones = torch.ones((H, W), dtype=torch.uint8, device="cuda:0")
    variants = ("render_tile", "moments", "masked_all_ones")
    times = {k: [] for k in variants}
    for i in range(args.warmup + args.reps):
        for k in variants:
            ctx.track_moments(k == "moments")
            ctx.reset_accum(W, H)
            ctx.synchronize()
            ctx.render_tile(p, mask=ones if k == "masked_all_ones" else None)
            ctx.synchronize()
            if i >= args.warmup:
                times[k].append(ctx.last_render_ms())
    ctx.track_moments(False)
    med = {k: float(np.median(v)) for k, v in times.items()}
    emit(dict(workload="overhead_c3_4k", width=W, height=H, camera_rays_per_pixel=16, max_bounce=10,
              **{f"ms_{k}": med[k] for k in variants},
              **{f"ms_spread_{k}": [float(np.min(v)), float(np.max(v))] for k, v in times.items()},
              overhead_moments=med["moments"] / med["render_tile"] - 1.0,
              overhead_masked_all_ones=med["masked_all_ones"] / med["render_tile"] - 1.0))
    del ones

    # ---- convergence: uniform passes against adaptive sampling at equal RMSE ---------------------------------------
    W, H = 1920, 1080
    center, half = mesh_box(sc)
    cam = framing(center, half, 0.0)
    base = dict(mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, seed=1)
    ctx.reset_accum(W, H)
    for b in range(0, args.ref_passes, 16):
        ctx.render_tile(rt.make_params(W, H, pass_begin=100000 + b, pass_count=min(16, args.ref_passes - b), **base), cam)
    ref = mean_image(ctx, W, H)

    uniform = []
    ctx.reset_accum(W, H)
    ctx.synchronize()
    dev_ms, t0, n = 0.0, time.perf_counter(), 0
    for stop in (4, 8, 16, 32, 64):
        ctx.render_tile(rt.make_params(W, H, pass_begin=n, pass_count=stop - n, **base), cam)
        dev_ms += ctx.last_render_ms()             # (synchronises)
        n = stop
        wall = (time.perf_counter() - t0) * 1e3
        uniform.append(dict(passes=n, device_ms=dev_ms, wall_ms=wall, camera_rays=W * H * n * 4, rmse=rmse(mean_image(ctx, W, H), ref)))
        t0 = time.perf_counter() - wall / 1e3       # (the readback for the RMSE is not part of the loop)
    emit(dict(workload="convergence_1080p", method="uniform", width=W, height=H, max_bounce=10, view="framed_front",
              ref_passes=args.ref_passes, points=uniform))
    u_rmse = np.array([u["rmse"] for u in uniform])
    u_rays = np.array([u["camera_rays"] for u in uniform], np.float64)
    u_ms = np.array([u["device_ms"] for u in uniform])

    mn, mx, ppr = 4, 64, 4
    for abs_tol, rel_tol in ((4e-3, 0.05), (2e-3, 0.02), (1e-3, 0.01), (5e-4, 0.005)):
        ctx.reset_accum(W, H)
        ctx.synchronize()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        # GpuContext.render_adaptive's loop, with each render call's device time
        ctx.track_moments(True)
        q = rt.make_params(W, H, pass_begin=0, pass_count=mn, **base)
        ctx.render_tile(q, cam)
        dev_ms = ctx.last_render_ms()
        rays, cursor, rounds = W * H * mn * 4, mn, 0
        while cursor < mx:
            mask, count = ctx.select_pixels(q, mn, mx, abs_tol, rel_tol)
            k = int(count.item())
            if k == 0:
                break
            step = min(ppr, mx - cursor)
            q.pass_begin, q.pass_count = cursor, step
            ctx.render_tile(q, cam, mask=mask)
            dev_ms += ctx.last_render_ms()
            rays += k * step * 4
            cursor += step
            rounds += 1
        ctx.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        ctx.track_moments(False)
        num = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)[..., 3]
        e = rmse(mean_image(ctx, W, H), ref)
        eq_rays, eq_ms = interp_loglog(e, u_rmse, u_rays), interp_loglog(e, u_rmse, u_ms)
        emit(dict(workload="convergence_1080p", method="adaptive", width=W, height=H, max_bounce=10, view="framed_front",
                  ref_passes=args.ref_passes, min_passes=mn, max_passes=mx, passes_per_round=ppr, abs_tol=abs_tol,
                  rel_tol=rel_tol, rounds=rounds, device_ms=dev_ms, wall_ms=wall, camera_rays=rays, rmse=e,
                  passes_mean=float(num.mean()), share_at_max=float((num >= mx).mean()),
                  share_at_min=float((num <= mn).mean()),
                  uniform_camera_rays_at_equal_rmse=eq_rays, uniform_device_ms_at_equal_rmse=eq_ms,
                  ray_ratio_at_equal_rmse=None if eq_rays is None else rays / eq_rays,
                  device_time_ratio_at_equal_rmse=None if eq_ms is None else dev_ms / eq_ms))
    ctx.close()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
