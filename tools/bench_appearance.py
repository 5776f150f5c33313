"""Cost of the appearance updates (GpuContext.update_materials / update_lights / update_texture, rt_gpu_update_materials /
_lights / _texture); one JSON line per workload.

   python tools/bench_appearance.py [--reps 20] [--warmup 3] [--frames 400] [--out FILE]

Workloads (unitychan, tests/scenes.py c3_unitychan, with texture slot 0 replaced by a 2048 x 2048 float texture so
that a full slot is the size of the reference's own textures):
  call_cost       per call: host time until the call returns (perf_counter) and device time of what it enqueued (CUDA
                  events on the calling stream around it; the stream is idle, so no frame is waited for), median of --reps:
                  a 64-node material batch over appended nodes, 8 lights, a full 2048 x 2048 slot from float texels and
                  from 4-channel 8-bit texels, and a 64 x 64 rectangle both ways.  The upload_scene of the same scene
                  (host time, it synchronises) is the line's reference.
  loop_4k         the 4-slot 4K frame loop of tools/bench_camera.py (3840 x 2160, one un-jittered ray per pixel, MaxBounceTimes
                  10), frames/s with one change per frame: nothing, a material node's colour, a 64 x 64 texel rectangle,
                  or upload_scene with the new colour (PATH); nothing, a moved light, or upload_scene with it (WHITTED).
                  --frames frames are timed after --warmup (--reps for the upload_scene loops, which take seconds).
The device name and power limit are read with nvidia-smi (query only) and go into every line.
"""
import argparse
import ctypes as C
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
from bench_queries import device_info  # noqa: E402

SLOT = 2048


class BigSlotScene:
    """unitychan's description with texture slot 0 of mesh 0 replaced by SLOT x SLOT float texels (host memory kept here)."""

    def __init__(self, sc):
        A = rt._abi
        d = sc.desc.contents
        self.sc = sc
        self.texels = np.random.default_rng(1).random((SLOT, SLOT, 4), dtype=np.float32)
        m = d.meshes[0]
        self.tex = (A.rt_texture * m.num_textures)()
        C.memmove(self.tex, m.textures, C.sizeof(self.tex))
        self.tex[0] = A.rt_texture(self.texels.ctypes.data_as(C.POINTER(C.c_float)), SLOT, SLOT, None, 0, None)
        self.meshes = (A.rt_mesh * d.num_meshes)()
        C.memmove(self.meshes, d.meshes, C.sizeof(self.meshes))
        self.meshes[0].textures = self.tex
        self.desc = A.rt_scene_desc()
        C.memmove(C.byref(self.desc), C.byref(d), C.sizeof(self.desc))
        self.desc.meshes = self.meshes

    def pointer(self):
        return C.pointer(self.desc)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=400, help="timed frames of a loop without uploads")
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
    big = BigSlotScene(sc)
    dev = torch.device("cuda", 0)
    A = rt._abi

    # ---- per call ------------------------------------------------------------------------------------------------
    ctx = rt.GpuContext(0)
    t = time.perf_counter()
    ctx.upload_scene(big.pointer())
    upload_ms = (time.perf_counter() - t) * 1e3
    n = big.desc.num_materials
    mats = [A.rt_material(rt._abi.RT_MAT_REFLECTIVE if k % 2 else rt._abi.RT_MAT_EMISSIVE, -1, -1, (0.5, 0.4, k / 64), 0.1)
            for k in range(64)]
    ctx.update_materials(mats, first=n)                     # appended once; the timed batches write over them
    lights = [(k % 2, (k * 0.5, 3.0, 2.0), (0.2, 0.2, 0.2)) for k in range(8)]
    full_f = torch.rand((SLOT, SLOT, 4), device=dev)
    full_8 = torch.randint(0, 256, (SLOT, SLOT, 4), dtype=torch.uint8, device=dev)
    rect_f = torch.rand((64, 64, 4), device=dev)
    rect_8 = torch.randint(0, 256, (64, 64, 4), dtype=torch.uint8, device=dev)
    calls = {
        "materials_64": lambda: ctx.update_materials(mats, first=n),
        "lights_8": lambda: ctx.update_lights(lights),
        "texture_full_2048_f32": lambda: ctx.update_texture(0, 0, full_f),
        "texture_full_2048_u8x4": lambda: ctx.update_texture(0, 0, full_8),
        "texture_rect_64_f32": lambda: ctx.update_texture(0, 0, rect_f, x=100, y=200),
        "texture_rect_64_u8x4": lambda: ctx.update_texture(0, 0, rect_8, x=100, y=200),
    }
    out = dict(workload="call_cost", slot=SLOT, upload_scene_host_ms=upload_ms)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for key, fn in calls.items():
        host, device = [], []
        for i in range(args.warmup + args.reps):
            torch.cuda.synchronize()
            ev0.record()
            t = time.perf_counter()
            fn()
            host_s = time.perf_counter() - t
            ev1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                host.append(host_s * 1e6)
                device.append(ev0.elapsed_time(ev1) * 1e3)
        out[f"{key}_host_us"] = float(np.median(host))
        out[f"{key}_device_us"] = float(np.median(device))
    emit(out)
    ctx.close()

    # ---- the 4-slot 4K loop with one change per frame ---------------------------------------------------------------
    W, H = 3840, 2160
    desc = big.desc
    node = next(k for k in range(desc.num_materials) if desc.materials[k].type == A.RT_MAT_DIFFUSE)
    base_rgb = list(desc.materials[node].rgb)
    res = {}
    for mode, hows in ((rt.RT_MODE_PATH, ("fixed", "material", "texture_rect_64", "upload_scene")),
                       (rt.RT_MODE_WHITTED, ("fixed", "light", "upload_scene"))):
        p = rt.make_params(W, H, mode=mode, max_bounce=10, pass_count=1, antialias=0, seed=1)
        for how in hows:
            ctx = rt.GpuContext(0)
            ctx.upload_scene(big.pointer())
            for s in range(4):
                ctx.set_frame_slot(s)
                ctx.reset_accum(W, H)
            for s in range(4):
                ctx.set_frame_slot(s)
                ctx.synchronize()
            timed = args.reps if how == "upload_scene" else args.frames
            t0 = None
            for i in range(args.warmup + timed):
                if i == args.warmup:
                    for s in range(4):
                        ctx.set_frame_slot(s)
                        ctx.synchronize()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                shade = 0.3 + 0.7 * (i % 8) / 8
                light = [(0, (2.0 * np.sin(i * 0.3), 3.0, 2.0 * np.cos(i * 0.3)), (1.0, 1.0, 1.0))]
                if how == "material":
                    m = A.rt_material.from_buffer_copy(desc.materials[node])
                    m.rgb[0] = shade
                    ctx.update_materials([m], first=node)
                elif how == "texture_rect_64":
                    ctx.update_texture(0, 0, rect_f if i % 2 else rect_8, x=(i * 64) % (SLOT - 64), y=128)
                elif how == "light":
                    ctx.update_lights(light)
                elif how == "upload_scene":
                    if mode == rt.RT_MODE_PATH:
                        desc.materials[node].rgb[0] = shade
                    else:
                        desc.lights[0].pos_or_dir[0] = light[0][1][0]
                        desc.lights[0].pos_or_dir[2] = light[0][1][2]
                    ctx.upload_scene(big.pointer())
                ctx.set_frame_slot(i % 4)
                p.pass_begin = i
                ctx.render_tile(p)
            for s in range(4):
                ctx.set_frame_slot(s)
                ctx.synchronize()
            torch.cuda.synchronize()
            res[(mode, how)] = timed / (time.perf_counter() - t0)
            ctx.close()
            desc.materials[node].rgb[0] = base_rgb[0]
    emit(dict(workload="loop_4k", width=W, height=H, slots=4, camera_rays_per_pixel=1, max_bounce=10, frames=args.frames,
              **{f"frames_per_s_{'path' if m == rt.RT_MODE_PATH else 'whitted'}_{h}": v for (m, h), v in res.items()}))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
