"""Replays the committed golden fixtures against
  * the plain-C restatement + the product's host scene layer     (CPU, always), and
  * the CUDA path through the C-ABI                                (-m gpu).
These do not need oracle/_ref at run time.  Which fixtures (tests_golden_common.golden):
  * tests/golden/*.npz, generated from the UNMODIFIED reference by tests/golden/make_golden.py, where the
    reference's meshes are staged (assets/_ref/Data); kat.npz (no mesh) always;
  * else tests/golden/standin/*.npz, the stand-in meshes (tests/standin_data.py) as the plain-C restatement
    rendered them (make_golden.py --standin): they pin later changes to what the project computed then,
    not to the reference."""
import hashlib
import os

import numpy as np
import pytest

import scenes
from conftest import GOLDEN_DIR, bits
from tests_golden_common import RENDERS, golden


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


# ---- CPU: restatement + host layer vs golden ------------------------------------------------------------
def test_kat_golden_port(port):
    g = golden("kat")
    a, t = port.kat_aabb(g["rays"], g["boxes"])
    np.testing.assert_array_equal(a, g["aabb_hit"])
    np.testing.assert_array_equal(bits(t), bits(g["aabb_tmin"]))
    for key, fn, prim in (("tri", port.kat_triangle, "tris"), ("sphere", port.kat_sphere, "spheres"),
                          ("plane", port.kat_plane, "planes"), ("capsule", port.kat_capsule, "caps")):
        f, o = fn(g["rays"], g[prim])
        np.testing.assert_array_equal(f, g[key + "_hit"])
        np.testing.assert_array_equal(bits(o), bits(g[key + "_out"]))
    np.testing.assert_array_equal(bits(port.kat_qrsqrt(g["x"])), bits(g["qrsqrt"]))
    np.testing.assert_array_equal(bits(port.kat_barycentric(g["pabc"])), bits(g["bary"]))
    np.testing.assert_array_equal(port.kat_display(g["rgb"]), g["display"])


@pytest.mark.parametrize("name", ["TorusKnot", "BlenderMonkey", "unitychan"])
def test_loader_bvh_primary_golden(rt, port, data_dir, name):
    g = golden(f"primary_{name}")
    sc = rt.Scene([("mesh", f"{data_dir}/{name}.obj", ("diffuse", scenes.WHITE))])
    assert sc.mesh_counts(0) == list(g["counts"])
    d = sc.mesh_dump(0)
    np.testing.assert_array_equal(sha(d["points"]), g["points_sha"])
    np.testing.assert_array_equal(sha(d["pidx"]), g["pidx_sha"])
    np.testing.assert_array_equal(sha(d["matid"]), g["matid_sha"])
    nodes, tris, shade = sc.flat_mesh(0)
    bounds = np.concatenate([nodes["bmin"], nodes["bmax"]], 1)
    np.testing.assert_array_equal(sha(bounds), g["bvh_bounds_sha"])
    np.testing.assert_array_equal(sha(nodes["escape"]), g["bvh_escape_sha"])
    leaf_tri = np.where(nodes["tri"] >= 0, tris["index"][np.maximum(nodes["tri"], 0)], -1).astype(np.int32)
    np.testing.assert_array_equal(sha(leaf_tri), g["bvh_tri_sha"])
    W, H = int(g["W"]), int(g["H"])
    p = rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=rt.RT_TRAVERSE_EXACT)
    o = port.render(sc.desc, p, want_primary=True)
    ids = o["ids"].reshape(-1, 2)
    np.testing.assert_array_equal(ids[:, 0], g["shape"].astype(np.int32))
    np.testing.assert_array_equal(ids[:, 1], g["tri"])
    np.testing.assert_array_equal(bits(o["dist"]).reshape(-1), bits(g["dist"]))
    assert o["counters"]["node_tests"] == int(g["node_tests"]) and o["counters"]["tri_tests"] == int(g["tri_tests"])


def test_textures_golden(rt, port, data_dir):
    g = golden("textures_unitychan")
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    assert int(g["count"]) == 8
    for k in range(8):
        px = sc.mesh_texture(0, int(g[f"tex{k}_slot"]))
        assert list(px.shape[:2]) == list(g[f"tex{k}_shape"])
        np.testing.assert_array_equal(sha(px), g[f"tex{k}_sha"])
        np.testing.assert_array_equal(bits(port.kat_texture_sample(px, g["uv"])), bits(g[f"tex{k}_samples"]))


def test_rays_default_scene_golden(rt, port, data_dir):
    g = golden("rays_default_scene")
    sc = rt.Scene(scenes.default_scene(data_dir))
    s, t, h = port.trace_rays(sc.desc, g["rays"])
    np.testing.assert_array_equal(s, g["shape"].astype(np.int32))
    np.testing.assert_array_equal(t, g["tri"])
    np.testing.assert_array_equal(bits(h), bits(g["hit"]))


@pytest.mark.parametrize("name", sorted(RENDERS))
def test_render_golden_port(rt, port, data_dir, name):
    g = golden(f"render_{name}")
    W, H, mode, bounce, aa, passes, seed, table_seed = [int(v) for v in g["params"]]
    sc = rt.Scene(getattr(scenes, RENDERS[name])(data_dir))
    if table_seed >= 0:
        sc.set_unit_vectors(seed=table_seed, count=0)
    pm = {0: rt.RT_MODE_PATH, 1: rt.RT_MODE_PREVIEW, 2: rt.RT_MODE_WHITTED}[mode]
    p = rt.make_params(W, H, mode=pm, max_bounce=bounce, antialias=aa, pass_count=passes, seed=seed, traverse=rt.RT_TRAVERSE_EXACT)
    o = port.render(sc.desc, p, nthreads=4, want_display=True)
    if mode == 1:
        # preview: the fixture's "accum" is the pass colour c (harness); accuBuffer itself stays untouched
        np.testing.assert_array_equal(bits(o["preview"][..., :3]), bits(g["accum"][..., :3]))
        assert not o["accum"].any()
    else:
        np.testing.assert_array_equal(bits(o["accum"]), bits(g["accum"]))
    np.testing.assert_array_equal(o["display"], g["display"])


# ---- GPU: the CUDA path vs golden ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["TorusKnot", "BlenderMonkey", "unitychan"])
def test_primary_golden_gpu(rt, gpu, data_dir, name):
    g = golden(f"primary_{name}")
    sc = rt.Scene([("mesh", f"{data_dir}/{name}.obj", ("diffuse", scenes.WHITE))])
    W, H = int(g["W"]), int(g["H"])
    gpu.upload_scene(sc)
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        gpu.reset_accum(W, H)
        gpu.reset_counters()
        gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=tr))
        ids = gpu.readback(rt.RT_READ_PRIMARY_IDS_I32X2, W, H).reshape(-1, 2)
        dist = gpu.readback(rt.RT_READ_PRIMARY_DIST_F32, W, H).reshape(-1)
        np.testing.assert_array_equal(ids[:, 0], g["shape"].astype(np.int32))
        np.testing.assert_array_equal(ids[:, 1], g["tri"])
        np.testing.assert_array_equal(bits(dist), bits(g["dist"]))
        if tr == rt.RT_TRAVERSE_EXACT:
            c = gpu.counters()
            assert c["node_tests"] == int(g["node_tests"]) and c["tri_tests"] == int(g["tri_tests"])


@pytest.mark.gpu
def test_rays_default_scene_golden_gpu(rt, gpu, data_dir):
    g = golden("rays_default_scene")
    sc = rt.Scene(scenes.default_scene(data_dir))
    gpu.upload_scene(sc)
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        s, t, h = gpu.trace_rays(g["rays"], tr)
        np.testing.assert_array_equal(s, g["shape"].astype(np.int32))
        np.testing.assert_array_equal(t, g["tri"])
        np.testing.assert_array_equal(bits(h), bits(g["hit"]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(RENDERS))
def test_render_golden_gpu(rt, gpu, data_dir, name):
    g = golden(f"render_{name}")
    W, H, mode, bounce, aa, passes, seed, table_seed = [int(v) for v in g["params"]]
    sc = rt.Scene(getattr(scenes, RENDERS[name])(data_dir))
    if table_seed >= 0:
        sc.set_unit_vectors(seed=table_seed, count=0)
    pm = {0: rt.RT_MODE_PATH, 1: rt.RT_MODE_PREVIEW, 2: rt.RT_MODE_WHITTED}[mode]
    gpu.upload_scene(sc)
    gpu.reset_accum(W, H)
    gpu.render_tile(rt.make_params(W, H, mode=pm, max_bounce=bounce, antialias=aa, pass_count=passes, seed=seed))
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    if mode == 1:
        assert not acc.any()                                   # UseBaseColor leaves accuBuffer alone
        acc = gpu.readback(rt.RT_READ_PREVIEW_RGBA_F32, W, H)  # w = 1 = the fixture's Num
    bad = (np.abs(acc - g["accum"]) > 1e-4).any(-1)
    if name == "default_path":
        # fuzzy reflections call sinf/cosf/acosf: CUDA's and glibc's differ in the last ulp, which can
        # steer a handful of paths onto another surface
        assert bad.mean() <= 2e-3
        assert abs(acc[..., :3].mean() - g["accum"][..., :3].mean()) <= 1e-3 * g["accum"][..., :3].mean()
    else:
        assert not bad.any()
        assert np.array_equal(bits(acc), bits(g["accum"]))
    disp = gpu.readback(rt.RT_READ_DISPLAY_ARGB8, W, H)
    ca = np.stack([(disp >> s) & 255 for s in (24, 16, 8, 0)], -1).astype(np.int32)
    cb = np.stack([(g["display"] >> s) & 255 for s in (24, 16, 8, 0)], -1).astype(np.int32)
    assert np.abs(ca - cb)[~bad].max() <= 1
