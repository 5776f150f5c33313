"""Times one rank's share of an N-GPU job on one GPU (tile_count=N, rank 0), no per-kernel events.
   python tools/rank_time.py [workload] [tiles] [repeats]   (knobs through the RT_* environment)"""
import os, sys, statistics
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import raytracerwin_b200 as rt
import bench

wl = sys.argv[1] if len(sys.argv) > 1 else "c4"
tiles = int(sys.argv[2]) if len(sys.argv) > 2 else 8
repeats = int(sys.argv[3]) if len(sys.argv) > 3 else 12
spec, W, H, passes, aa, bounce, mode, desc = bench.build_spec(wl)
scene = rt.Scene(spec)
pm = {"path": rt.RT_MODE_PATH, "preview": rt.RT_MODE_PREVIEW, "whitted": rt.RT_MODE_WHITTED}[mode]
if mode == "path": scene.set_unit_vectors(0, 0)
ctx = rt.GpuContext(0)
ctx.upload_scene(scene)
variants = os.environ.get("RT_VARIANTS", "").split(";")
for v in variants:
    os.environ.pop("RT_SAMPLE_BUDGET_MB", None)
    os.environ.update(RT_LONG_LIMIT="2048", RT_SMALL_ROUND="24000", RT_LONG_GROUP_N="32", RT_THIN_COUNT="200000", RT_THIN_LIMIT="256", RT_PIPES_N="4", RT_PACKET_ROUNDS="-1", RT_PACKET_PROBE="24", RT_PACKET_MIN_LANES="10")
    for kv in v.split():
        k, x = kv.split("="); os.environ[k] = x
    ctx.set_pipes(int(os.environ.get("RT_PIPES_N", "4")))
    ctx.set_tuning(32, 28, 18, 0)
    tk = dict(tile_size=32, tile_count=tiles, tile_rank=0) if tiles > 1 else {}
    p = rt.make_params(W, H, mode=pm, max_bounce=bounce, pass_count=passes, antialias=aa, seed=0, **tk)
    ms = []
    for i in range(repeats + 3):
        ctx.reset_accum(W, H)
        ctx.render_tile(p)
        ms.append(ctx.last_render_ms())
    ms = ms[3:]
    print(f"{wl} tiles={tiles} [{v}] median {statistics.median(ms):.3f} ms  min {min(ms):.3f}  max {max(ms):.3f}", flush=True)
ctx.close()
