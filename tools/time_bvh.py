"""Host vs device build of the reference's tree for the bench scenes (SURVEY 8f-1).  python tools/time_bvh.py [c3 c5s c5]
Uses bench.py's generated stand-ins when the reference's meshes are not staged."""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import raytracerwin_b200 as rt
import bench
if not os.path.isdir(bench.DATA):                  # the reference's meshes are not staged: bench.py's stand-ins
    import standin_data
    bench.DATA = standin_data.write(os.path.join(bench.scratch_dir(), "Data"))
ctx = rt.GpuContext(0)
for wl in (sys.argv[1:] or ["c3", "c5s", "c5"]):
    spec, *_ = bench.build_spec(wl)
    t0 = time.perf_counter(); sc = rt.Scene(spec); t_load = time.perf_counter() - t0
    d = sc.mesh_dump(0)
    n = len(d["pidx"]) // 3
    # host build alone: the same arrays through rt_host_add_mesh_arrays (copy + build + shading records)
    t0 = time.perf_counter()
    sc2 = rt.Scene(); sc2.add_mesh_arrays(d["points"], d["pidx"], material=("diffuse", (1, 1, 1)))
    t_host = time.perf_counter() - t0
    nodes, tris, _ = sc.flat_mesh(0)
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        gn, gt, depth, ms = ctx.build_bvh(d["points"], d["pidx"])
        wall = time.perf_counter() - t0
        best = ms if best is None else min(best, ms)
    same = gn.tobytes() == nodes.tobytes() and gt.tobytes() == tris.tobytes()
    print(json.dumps({"scene": wl, "triangles": n, "depth": depth, "obj_load_total_s": t_load, "host_build_s": t_host,
                      "gpu_build_device_ms": best, "gpu_build_wall_s_incl_copies": wall, "bit_identical": same,
                      "speedup_device_vs_host": t_host * 1e3 / best}), flush=True)
