"""Cost and gain of the guided denoiser (RT_MODE_GUIDES, rt_gpu_denoise); one JSON line per workload.

   python tools/bench_denoise.py [--reps 20] [--warmup 5] [--ref-passes 256] [--out FILE]

Workloads (unitychan, tests/scenes.py c3_unitychan, on the close front view of tools/bench_camera.py, framing(yaw = 0)):
  time_<size>         device time of one GpuContext.denoise (use_albedo, use_variance, argb on) at 1920 x 1080 and
                      3840 x 2160 for levels 1..5: CUDA events around the call on the current torch stream, median of
                      --reps after --warmup, the output buffers allocated once.  bytes = the records each kernel reads
                      and writes once (level 0: 76 B read, 36 B written per pixel; a level: 36 B read, 16 B written;
                      the last one also reads accum and preview and writes rgba and argb), floor_ms = bytes at 7.7 TB/s.
                      A 1080p frame's records (~110 MB) fit the 126 MB L2, so there the floor is not a bound.
                      Also the device time of the RT_MODE_GUIDES render (rt_gpu_last_render_ms) at each size.
  quality_1080p       PATH, MaxBounceTimes 10, antialiased, at 1920 x 1080.  Reference: the mean of --ref-passes passes of
                      other pass indices.  For N = 4 .. 64 passes (moments tracked, a PREVIEW pass, a GUIDES render): RMSE
                      of the raw mean and of the denoised frame (levels 5, albedo and variance, defaults otherwise)
                      against the reference, and the uniform pass count and render device time at which the raw mean
                      reaches each denoised RMSE (log-log interpolation over raw N = 4 .. 256; null outside).
The device name and power limit are read with nvidia-smi (query only) and go into every line.
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
from bench_adaptive import interp_loglog, mean_image, rmse  # noqa: E402
from bench_camera import framing, mesh_box  # noqa: E402
from bench_queries import device_info  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def denoise_bytes(npix, levels):
    return npix * ((76 + 36) + levels * (36 + 16) + (16 + 16) + (16 + 4))


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ref-passes", type=int, default=256)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, power = device_info()
    scratch = tempfile.TemporaryDirectory(prefix="rtb200_bd_")
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
    center, half = mesh_box(sc)
    cam = framing(center, half, 0.0)
    base = dict(mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, seed=1)
    stream = torch.cuda.current_stream()

    # ---- device time per call ---------------------------------------------------------------------------------------
    for W, H in ((1920, 1080), (3840, 2160)):
        ctx.reset_accum(W, H)
        ctx.track_moments(True)
        ctx.render_tile(rt.make_params(W, H, pass_count=4, **base), cam)
        ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PREVIEW, seed=1), cam)
        guides_ms = []
        for _ in range(5):
            ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_GUIDES), cam)
            guides_ms.append(ctx.last_render_ms())
        ctx.synchronize()
        out = torch.empty((H, W, 4), dtype=torch.float32, device="cuda:0")
        pix_out = None
        per_level = {}
        for levels in range(1, 6):
            def call():
                return ctx.denoise(levels=levels, use_albedo=True, use_variance=True, out=out, argb=True)
            for _ in range(args.warmup):
                _, pix_out = call()
            times = []
            for _ in range(args.reps):
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record(stream)
                call()
                t1.record(stream)
                t1.synchronize()
                times.append(t0.elapsed_time(t1))
            med = float(np.median(times))
            b = denoise_bytes(W * H, levels)
            per_level[levels] = dict(ms=med, ms_spread=[float(np.min(times)), float(np.max(times))], bytes=b,
                                     floor_ms=b / HBM_BYTES_PER_S * 1e3, floor_share=b / HBM_BYTES_PER_S * 1e3 / med)
        ctx.track_moments(False)
        emit(dict(workload=f"time_{H}p" if H != 2160 else "time_4k", width=W, height=H, launches_per_call="1 + levels",
                  guides_render_ms=float(np.median(guides_ms)), levels=per_level))
        del out, pix_out

    # ---- quality: raw and denoised RMSE against a long reference ------------------------------------------------------
    W, H = 1920, 1080
    ctx.reset_accum(W, H)
    for b in range(0, args.ref_passes, 16):
        ctx.render_tile(rt.make_params(W, H, pass_begin=100000 + b, pass_count=min(16, args.ref_passes - b), **base), cam)
    ref = mean_image(ctx, W, H)
    ctx.reset_accum(W, H)
    ctx.track_moments(True)
    ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PREVIEW, seed=1), cam)
    ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_GUIDES), cam)
    ctx.synchronize()
    raw, den, dev_ms, n = [], [], 0.0, 0
    for stop in (4, 8, 16, 32, 64, 128, 256):
        ctx.render_tile(rt.make_params(W, H, pass_begin=n, pass_count=stop - n, **base), cam)
        dev_ms += ctx.last_render_ms()
        n = stop
        raw.append(dict(passes=n, render_device_ms=dev_ms, rmse=rmse(mean_image(ctx, W, H), ref)))
        if n <= 64:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            img = ctx.denoise(levels=5, use_albedo=True, use_variance=True)
            t1.record(stream)
            t1.synchronize()
            den.append(dict(passes=n, render_device_ms=dev_ms, denoise_ms=t0.elapsed_time(t1),
                            rmse=rmse(img[..., :3].cpu().numpy().astype(np.float64), ref)))
    ctx.track_moments(False)
    r_rmse = np.array([r["rmse"] for r in raw])
    r_pass = np.array([r["passes"] for r in raw], np.float64)
    r_ms = np.array([r["render_device_ms"] for r in raw])
    for d in den:
        d["raw_rmse"] = next(r["rmse"] for r in raw if r["passes"] == d["passes"])
        d["raw_passes_at_equal_rmse"] = interp_loglog(d["rmse"], r_rmse, r_pass)
        d["raw_render_device_ms_at_equal_rmse"] = interp_loglog(d["rmse"], r_rmse, r_ms)
    emit(dict(workload="quality_1080p", width=W, height=H, max_bounce=10, view="framed_front", ref_passes=args.ref_passes,
              denoise=dict(levels=5, use_albedo=True, use_variance=True, normal_log2=7, sigma_lum=4.0, sigma_depth=0.1,
                           lum_floor=0.02),
              raw=raw, denoised=den))
    ctx.close()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
