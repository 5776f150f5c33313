"""BASELINE configs[4] at test scale: a generated OBJ of translated copies (tools/make_c5.py) through the ordinary
loader — deeper tree, many more nodes per ray.  CPU: host loader/BVH + restatement vs the reference.  GPU: CUDA
path vs the restatement at a larger copy count."""
import os
import sys

import numpy as np
import pytest

from conftest import DATA_DIR, ROOT, bits

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_c5  # noqa: E402

WHITE = (1.0, 1.0, 1.0)


def test_generated_grid_cpu_vs_reference(tmp_path, rt, port, ref, data_dir):
    out = str(tmp_path / "torus_48.obj")
    make_c5.main(os.path.join(data_dir, "TorusKnot.obj"), out, 48)
    spec = [("mesh", out, ("reflective", (0.8, 0.8, 0.8), 0.0))]
    sc = rt.Scene(spec)
    rs = ref.build_scene(spec)
    assert sc.mesh_counts(0) == ref.mesh_counts(rs, 0)
    assert sc.mesh_counts(0)[3] == 48 * 1200
    bounds, escape, tri, verts = ref.mesh_bvh(rs, 0)
    nodes, tris, shade = sc.flat_mesh(0)
    np.testing.assert_array_equal(bits(nodes["bmin"]), bits(bounds[:, :3]))
    np.testing.assert_array_equal(nodes["escape"], escape)
    W, H = 320, 180
    r = ref.trace_primary(rs, W, H)
    o = port.render(sc.desc, rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=rt.RT_TRAVERSE_EXACT), nthreads=4, want_primary=True)
    ids = o["ids"].reshape(-1, 2)
    np.testing.assert_array_equal(ids[:, 1], r["tri"])
    np.testing.assert_array_equal(bits(o["dist"]).reshape(-1), bits(r["dist"]))
    assert (r["tri"] >= 0).mean() > 0.15                      # the grid fills the frame
    assert o["counters"]["node_tests"] == r["node_tests"]
    ref.free_scene(rs)


@pytest.mark.gpu
def test_generated_grid_gpu(tmp_path, rt, gpu, port, data_dir):
    out = str(tmp_path / "unitychan_12.obj")
    make_c5.main(os.path.join(data_dir, "unitychan.obj"), out, 12)          # 193 k triangles, textured
    spec = [("mesh", out, ("blend", ("reflective", WHITE, 0.2), ("diffuse", WHITE), 1.0))]
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=1, count=1 << 20)
    one = rt.Scene([("mesh", os.path.join(data_dir, "unitychan.obj"), ("diffuse", WHITE))]).mesh_counts(0)[3]
    if data_dir == DATA_DIR:
        assert one == 16056                                                   # the reference's unitychan
    assert sc.mesh_counts(0)[3] == 12 * one
    gpu.upload_scene(sc)
    W, H = 640, 360
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        p = rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=tr)
        gpu.reset_accum(W, H)
        gpu.reset_counters()
        gpu.render_tile(p)
        ids = gpu.readback(rt.RT_READ_PRIMARY_IDS_I32X2, W, H)
        dist = gpu.readback(rt.RT_READ_PRIMARY_DIST_F32, W, H)
        p.traverse = rt.RT_TRAVERSE_EXACT
        o = port.render(sc.desc, p, nthreads=8, want_primary=True)
        np.testing.assert_array_equal(ids, o["ids"])
        np.testing.assert_array_equal(bits(dist), bits(o["dist"]))
        if tr == rt.RT_TRAVERSE_EXACT:
            assert gpu.counters()["node_tests"] == o["counters"]["node_tests"]
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=6, antialias=1, pass_count=1, seed=2)
    gpu.reset_accum(W, H)
    gpu.render_tile(p)
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    o = port.render(sc.desc, p, nthreads=8)
    assert np.array_equal(bits(acc), bits(o["accum"]))
