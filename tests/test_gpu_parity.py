"""GPU parity tests: the CUDA path, called through the C-ABI (include/rt_gpu.h), against
  * the UNMODIFIED reference compiled into oracle/_ref/libref_oracle.so (when present), and
  * the plain-C restatement oracle/librt_oracle.so (always),
on the same scenes, cameras and counter-RNG seeds.

Bars (BASELINE.json north_star): primary (shape, triangle) ids and Distance bits EXACT; shaded linear
RGB within 1e-4 per channel on deterministic paths; stochastic paths: the shared counter RNG makes
the two sides draw identical numbers, so the bar here is stricter than a statistical one —
>= 99.9 % of pixels within 1e-4 and the image mean within 0.1 % (the residue is CUDA-vs-glibc
sinf/cosf/acosf ulps in fuzzy reflections steering a path to a different surface).
"""
import numpy as np
import pytest

import scenes
from conftest import bits, is_reference, same_bits

pytestmark = pytest.mark.gpu

TOL = 1e-4


def gpu_render(rt, gpu, scene, W, H, **kw):
    p = rt.make_params(W, H, **kw)
    gpu.upload_scene(scene)
    gpu.reset_accum(W, H)
    gpu.reset_counters()
    gpu.render_tile(p)
    out = dict(accum=gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H),
               display=gpu.readback(rt.RT_READ_DISPLAY_ARGB8, W, H),
               counters=gpu.counters())
    if kw.get("mode") == rt.RT_MODE_PREVIEW:
        out["preview"] = gpu.readback(rt.RT_READ_PREVIEW_RGBA_F32, W, H)
    if kw.get("mode") == rt.RT_MODE_PRIMARY:
        out["ids"] = gpu.readback(rt.RT_READ_PRIMARY_IDS_I32X2, W, H)
        out["dist"] = gpu.readback(rt.RT_READ_PRIMARY_DIST_F32, W, H)
    return out, p


def assert_display_close(a, b):
    """ARGB8: CUDA powf vs glibc powf may differ by one code value at a rounding boundary."""
    ca = np.stack([(a >> s) & 255 for s in (24, 16, 8, 0)], -1).astype(np.int32)
    cb = np.stack([(b >> s) & 255 for s in (24, 16, 8, 0)], -1).astype(np.int32)
    assert np.abs(ca - cb).max() <= 1


# ---------------------------------------------------------------------------------------------------
# T0: primary hits, bit exact, on the three reference meshes at their config resolutions
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,W,H", [("TorusKnot", 640, 480), ("BlenderMonkey", 1920, 1080), ("unitychan", 1920, 1080)])
@pytest.mark.parametrize("traverse", ["exact", "culled"])
def test_primary_ids_bit_exact_vs_reference(rt, gpu, ref, data_dir, name, W, H, traverse):
    spec = [("mesh", f"{data_dir}/{name}.obj", ("diffuse", scenes.WHITE))]
    sc = rt.Scene(spec)
    tr = rt.RT_TRAVERSE_EXACT if traverse == "exact" else rt.RT_TRAVERSE_CULLED
    out, _ = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PRIMARY, traverse=tr)
    rs = ref.build_scene(spec)
    r = ref.trace_primary(rs, W, H)
    assert r["mismatches"] == 0
    ids = out["ids"].reshape(-1, 2)
    assert (r["shape"] >= 0).sum() > 1000
    np.testing.assert_array_equal(ids[:, 0], r["shape"])
    np.testing.assert_array_equal(ids[:, 1], r["tri"])
    np.testing.assert_array_equal(bits(out["dist"]).reshape(-1), bits(r["dist"]))
    c = out["counters"]
    assert c["rays"] == W * H and c["camera_rays"] == W * H
    if traverse == "exact":
        # the device walks exactly the nodes / triangles the reference walks
        assert c["node_tests"] == r["node_tests"] and c["tri_tests"] == r["tri_tests"]
        assert c["node_visits"] == r["node_tests"] and c["tri_visits"] == r["tri_tests"]
    else:
        assert c["node_visits"] <= r["node_tests"] and c["tri_visits"] <= r["tri_tests"]
    ref.free_scene(rs)


def test_primary_default_scene_vs_port(rt, gpu, port, data_dir):
    """All shape classes + the stale-hit-field quirk: ids, distance and the 11 hit floats."""
    sc = rt.Scene(scenes.default_scene(data_dir))
    W, H = 800, 800
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        out, p = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PRIMARY, traverse=tr)
        p.traverse = rt.RT_TRAVERSE_EXACT
        o = port.render(sc.desc, p, nthreads=8, want_primary=True)
        np.testing.assert_array_equal(out["ids"], o["ids"])
        np.testing.assert_array_equal(bits(out["dist"]), bits(o["dist"]))


def random_rays(n, seed, scale=3.0):
    rng = np.random.default_rng(seed)
    o = rng.normal(size=(n, 3)).astype(np.float32) * np.float32(scale)
    tgt = rng.normal(size=(n, 3)).astype(np.float32) * np.float32(0.8)
    d = tgt - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    dist = rng.choice(np.array([1000.0, 10.0, 3.0, 0.5], np.float32), size=n)
    rays = np.concatenate([o, d.astype(np.float32), dist[:, None]], 1).astype(np.float32)
    # axis-aligned and zero-component directions exercise the disabled-slab quirk (Appendix A2)
    k = n // 16
    rays[:k, 3:6] = 0.0
    rays[:k, 3 + (np.arange(k) % 3)] = np.where(rng.random(k) < 0.5, -1.0, 1.0)
    rays[k:2 * k, 4] = 0.0
    nrm = np.linalg.norm(rays[k:2 * k, 3:6], axis=1, keepdims=True)
    rays[k:2 * k, 3:6] /= np.where(nrm == 0, 1, nrm)
    return rays


@pytest.mark.parametrize("scene_name", ["default_scene", "deterministic_mix", "c3_unitychan"])
def test_trace_rays_bit_exact(rt, gpu, port, ref, data_dir, scene_name):
    """Incoherent rays from everywhere (inside boxes, behind, short): every hit field bit for bit."""
    spec = getattr(scenes, scene_name)(data_dir)
    sc = rt.Scene(spec)
    gpu.upload_scene(sc)
    rays = random_rays(200_000, 7)
    ps, pt, ph = port.trace_rays(sc.desc, rays)
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        gs, gt, gh = gpu.trace_rays(rays, tr)
        np.testing.assert_array_equal(gs, ps)
        np.testing.assert_array_equal(gt, pt)
        np.testing.assert_array_equal(bits(gh), bits(ph))
    assert (ps >= 0).mean() > 0.05
    # and the restatement agrees with the reference itself on the same rays
    if is_reference(ref, "restatement vs reference ray casts"):
        rs = ref.build_scene(spec)
        sub = rays[:20_000]
        s2, t2, h2 = ref.trace_rays(rs, sub)
        np.testing.assert_array_equal(ps[:20_000], s2)
        np.testing.assert_array_equal(pt[:20_000], t2)
        np.testing.assert_array_equal(bits(ph[:20_000]), bits(h2))
        ref.free_scene(rs)


# ---------------------------------------------------------------------------------------------------
# T1: deterministic shading within 1e-4 (in practice: bit exact)
# ---------------------------------------------------------------------------------------------------
def test_c1_whitted_vs_reference(rt, gpu, ref, data_dir):
    spec = scenes.c1_torusknot(data_dir)
    sc = rt.Scene(spec)
    W, H = 640, 480
    out, _ = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_WHITTED, antialias=0, pass_count=1)
    rs = ref.build_scene(spec)
    r = ref.render(rs, W, H, mode=2, antialias=0, pass_count=1, nthreads=8, want_display=True)
    np.testing.assert_allclose(out["accum"], r["accum"], atol=TOL, rtol=0)
    assert np.array_equal(bits(out["accum"]), bits(r["accum"]))      # stronger than asked
    assert_display_close(out["display"], r["display"])
    hits = (out["accum"][..., :3].sum(-1) == 0).sum()
    assert hits > 0                                                    # some pixels are in shadow / unlit
    assert out["counters"]["shadow_rays"] == r["shadow_rays"]
    ref.free_scene(rs)


@pytest.mark.parametrize("scene_name,bounce", [("c2_monkey", 5), ("c2_monkey_null", 5), ("deterministic_mix", 10)])
def test_deterministic_paths_vs_reference(rt, gpu, ref, data_dir, scene_name, bounce):
    spec = getattr(scenes, scene_name)(data_dir)
    sc = rt.Scene(spec)
    W, H = (1920, 1080) if scene_name == "c2_monkey" else (640, 360)
    rs = ref.build_scene(spec)
    r = ref.render(rs, W, H, mode=0, max_bounce=bounce, antialias=0, pass_count=1, nthreads=8, want_display=True)
    for tr in (rt.RT_TRAVERSE_CULLED, rt.RT_TRAVERSE_EXACT):
        out, _ = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PATH, max_bounce=bounce, antialias=0, pass_count=1, traverse=tr)
        np.testing.assert_allclose(out["accum"], r["accum"], atol=TOL, rtol=0)
        assert_display_close(out["display"], r["display"])
    ref.free_scene(rs)


def test_preview_pass_vs_reference(rt, gpu, ref, data_dir):
    """RenderOption.UseBaseColor (RayTracerScene.cpp:54-61) on the textured mesh: texture sampling parity."""
    spec = scenes.c3_unitychan(data_dir)
    sc = rt.Scene(spec)
    W, H = 960, 540
    out, _ = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PREVIEW, antialias=1, pass_count=1, seed=3)
    rs = ref.build_scene(spec)
    r = ref.render(rs, W, H, mode=1, antialias=1, pass_count=1, seed=3, nthreads=8, want_display=True)
    # (the harness returns the pass colour c in its accum argument; the product keeps it apart, see below)
    np.testing.assert_allclose(out["preview"][..., :3], r["accum"][..., :3], atol=TOL, rtol=0)
    assert np.array_equal(bits(out["preview"][..., :3]), bits(r["accum"][..., :3]))
    assert_display_close(out["display"], r["display"])
    ref.free_scene(rs)
    # UseBaseColor writes bitcolor only: accuBuffer is untouched (RayTracerProgram.cpp:175-180)
    assert not out["accum"].any()


def test_preview_then_passes_without_reset(rt, gpu, port, data_dir):
    """The reference's Run(): a preview pass, then N accumulation passes on the same buffers with no reset in
    between (RayTracerProgram.cpp:291-327).  The preview must leave accuBuffer (sum and Num) alone."""
    spec = scenes.c3_unitychan(data_dir)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=0, count=1 << 20)
    W, H = 320, 180
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=6, antialias=1, seed=4)
    alone, _ = gpu_render(rt, gpu, sc, W, H, pass_count=3, **kw)
    gpu.reset_accum(W, H)
    gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PREVIEW, antialias=1, pass_count=1, seed=4))
    shown = gpu.readback(rt.RT_READ_DISPLAY_ARGB8, W, H)
    for k in range(3):
        gpu.render_tile(rt.make_params(W, H, pass_begin=k, pass_count=1, **kw))
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert np.array_equal(bits(acc), bits(alone["accum"]))
    assert (acc[..., 3] == 3).all()
    np.testing.assert_array_equal(gpu.readback(rt.RT_READ_DISPLAY_ARGB8, W, H), alone["display"])
    assert (shown != alone["display"]).any()                         # the preview did show something else
    # and the restatement behaves the same way
    a = np.zeros((H, W, 4), np.float32)
    port.render(sc.desc, rt.make_params(W, H, mode=rt.RT_MODE_PREVIEW, antialias=1, pass_count=1, seed=4), nthreads=8, accum=a)
    assert not a.any()
    o = port.render(sc.desc, rt.make_params(W, H, pass_count=3, **kw), nthreads=8, accum=a)
    assert np.array_equal(bits(o["accum"]), bits(acc))


# ---------------------------------------------------------------------------------------------------
# T2: stochastic paths under the shared counter RNG
# ---------------------------------------------------------------------------------------------------
def stochastic_check(g, r):
    g3, r3 = g[..., :3], r[..., :3]
    np.testing.assert_array_equal(g[..., 3], r[..., 3])
    bad = (np.abs(g3 - r3) > TOL).any(-1)
    frac = bad.mean()
    mean_err = abs(g3.mean() - r3.mean()) / max(r3.mean(), 1e-9)
    return frac, mean_err


def test_c3_unitychan_stochastic_vs_reference(rt, gpu, ref, data_dir):
    """C3 at quarter resolution, full 16 camera rays / pixel (4 passes x 4 jittered), MaxBounceTimes 10."""
    spec = scenes.c3_unitychan(data_dir)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=0, count=0)
    ref.init_unit_vectors(0)
    if is_reference(ref, "unit-vector table"):
        np.testing.assert_array_equal(bits(ref.unit_vector_table()[:4096]),
                                      bits(np.ctypeslib.as_array(sc.desc.contents.unit_vectors, (4096 * 3,)).reshape(-1, 3)))
    W, H = 480, 270
    out, _ = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, pass_count=4, seed=0)
    rs = ref.build_scene(spec)
    r = ref.render(rs, W, H, mode=0, max_bounce=10, antialias=1, pass_count=4, seed=0, nthreads=8)
    frac, mean_err = stochastic_check(out["accum"], r["accum"])
    assert frac <= 1e-3, frac
    assert mean_err <= 1e-3, mean_err
    # Diffuse only (Blend factor 1.0): no libm on the path, so the match is in fact exact
    assert np.array_equal(bits(out["accum"]), bits(r["accum"]))
    ref.free_scene(rs)


def test_default_scene_stochastic_vs_port_and_reference(rt, gpu, port, ref, data_dir):
    """All seven material classes incl. fuzzy reflection (sinf/cosf/acosf) and Combine order."""
    spec = scenes.default_scene(data_dir)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=5, count=0)
    W, H = 400, 400
    out, p = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, pass_count=2, seed=11)
    o = port.render(sc.desc, p, nthreads=8)
    frac, mean_err = stochastic_check(out["accum"], o["accum"])
    assert frac <= 2e-3, frac
    assert mean_err <= 1e-3, mean_err
    ref.init_unit_vectors(5)
    rs = ref.build_scene(spec)
    r = ref.render(rs, W, H, mode=0, max_bounce=10, antialias=1, pass_count=2, seed=11, nthreads=8)
    frac, mean_err = stochastic_check(out["accum"], r["accum"])
    assert frac <= 2e-3, frac
    assert mean_err <= 1e-3, mean_err
    assert out["counters"]["rays"] > out["counters"]["camera_rays"]
    ref.free_scene(rs)


def test_default_scene_statistical_contract(rt, gpu, ref, data_dir):
    """SURVEY.md 8(c) tier T2 as written, on the one scene whose paths are NOT bit-reproducible (fuzzy reflection
    calls sinf / cosf / acosf, whose CUDA and glibc results differ in the last ulp and can steer a path elsewhere):
    n independent passes on both sides, per-pixel means and variances, then
      |mean_gpu - mean_cpu| <= 4 * sqrt((s2_cpu + s2_gpu) / n) for >= 99.9 % of pixels (per channel), and
      image-mean relative error < 0.5 %, and no spatial structure in the residual (its block means are as small
      as independent noise allows)."""
    spec = scenes.default_scene(data_dir)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=5, count=0)
    ref.init_unit_vectors(5)
    rs = ref.build_scene(spec)
    W, H, n = 200, 200, 12
    gpu.upload_scene(sc)
    g = np.zeros((n, H, W, 3), np.float64)
    c = np.zeros((n, H, W, 3), np.float64)
    for k in range(n):
        gpu.reset_accum(W, H)
        gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, pass_begin=k, pass_count=1, seed=31))
        g[k] = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)[..., :3]
        c[k] = ref.render(rs, W, H, mode=0, max_bounce=10, antialias=1, pass_begin=k, pass_count=1, seed=31, nthreads=8)["accum"][..., :3]
    ref.free_scene(rs)
    gm, cm = g.mean(0), c.mean(0)
    bound = 4.0 * np.sqrt((g.var(0, ddof=1) + c.var(0, ddof=1)) / n)
    ok = np.abs(gm - cm) <= bound + 1e-6              # (+1e-6: pixels both sides render identically have zero variance)
    assert ok.all(-1).mean() >= 0.999, ok.all(-1).mean()
    assert abs(gm.mean() - cm.mean()) / cm.mean() < 5e-3
    # residual block means: a systematic difference (a wrong material, a shifted texture) would show up as blocks far
    # outside what the per-pixel spread predicts
    res = (gm - cm).mean(-1)
    blocks = res.reshape(H // 20, 20, W // 20, 20).mean((1, 3))
    spread = np.sqrt(((g.var(0, ddof=1) + c.var(0, ddof=1)) / n).mean(-1)).reshape(H // 20, 20, W // 20, 20).mean((1, 3)) / 20.0
    assert (np.abs(blocks) <= 6.0 * spread + 1e-4).all()
    # most pixels are in fact identical: the shared counter RNG makes both sides draw the same numbers
    assert (np.abs(gm - cm) <= TOL).all(-1).mean() >= 0.99


# ---------------------------------------------------------------------------------------------------
# size-independent properties at full config sizes
# ---------------------------------------------------------------------------------------------------
def test_c3_full_size_exact_equals_culled_and_tiles(rt, gpu, data_dir):
    """1920x1080, 16 camera rays/pixel: (i) culled == exact traversal bit for bit; (ii) the frame
    assembled from 4 tile-interleaved 'ranks' (pack -> unpack) == the single-context frame;
    (iii) splitting the passes over two calls == one call (accumulation order is fixed)."""
    import torch
    spec = scenes.c3_unitychan(data_dir)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=0, count=0)
    W, H = 1920, 1080
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, seed=0)
    full, _ = gpu_render(rt, gpu, sc, W, H, pass_count=4, traverse=rt.RT_TRAVERSE_CULLED, **kw)
    exact, _ = gpu_render(rt, gpu, sc, W, H, pass_count=4, traverse=rt.RT_TRAVERSE_EXACT, **kw)
    assert np.array_equal(bits(full["accum"]), bits(exact["accum"]))
    assert full["counters"]["rays"] == exact["counters"]["rays"]
    assert full["counters"]["node_visits"] < exact["counters"]["node_visits"]
    # (iii)
    gpu.reset_accum(W, H)
    gpu.render_tile(rt.make_params(W, H, pass_begin=0, pass_count=1, **kw))
    gpu.render_tile(rt.make_params(W, H, pass_begin=1, pass_count=3, **kw))
    split = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert np.array_equal(bits(split), bits(full["accum"]))
    # (ii) four ranks emulated one after another on this GPU, exchanged through dense buffers
    n = 4
    root = np.zeros((H, W, 4), np.float32)
    dense = []
    for r in range(n):
        p = rt.make_params(W, H, pass_count=4, tile_size=32, tile_count=n, tile_rank=r, **kw)
        gpu.reset_accum(W, H)
        gpu.render_tile(p)
        cnt = rt.owned_pixels(W, H, 32, n, r)
        buf = torch.empty((cnt, 4), dtype=torch.float32, device="cuda:0")
        gpu.pack_owned(p, buf.data_ptr(), buf.numel() * 4)
        gpu.synchronize()
        dense.append((p, buf))
    assert sum(b.shape[0] for _, b in dense) == W * H
    gpu.reset_accum(W, H)
    for r, (p, buf) in enumerate(dense):
        gpu.unpack_owned(p, r, buf.data_ptr(), buf.numel() * 4)
    gpu.synchronize()
    root = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert np.array_equal(bits(root), bits(full["accum"]))


def test_task_ranges_and_edge_cases(rt, gpu, port, data_dir):
    """RenderThreadTask ranges (inclusive, 10 rows each), ragged ranges, empty ranges, 1x1 frames,
    odd sizes, max_bounce 0/1."""
    spec = scenes.deterministic_mix(data_dir)
    sc = rt.Scene(spec)
    gpu.upload_scene(sc)
    W, H = 333, 117
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=6, antialias=0)
    whole, p = gpu_render(rt, gpu, sc, W, H, **kw)
    o = port.render(sc.desc, p, nthreads=8)
    assert np.array_equal(bits(whole["accum"]), bits(o["accum"]))
    # the reference's task split: 10 rows per task
    gpu.reset_accum(W, H)
    for row in range(0, H, 10):
        start, end = row * W, min((row + 10) * W - 1, W * H - 1)
        gpu.render_tile(rt.make_params(W, H, start=start, end=end, **kw))
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(whole["accum"]))
    # ragged range inside rows; pixels outside stay untouched
    gpu.reset_accum(W, H)
    s, e = 5 * W + 17, 9 * W + 3
    gpu.render_tile(rt.make_params(W, H, start=s, end=e, **kw))
    part = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).reshape(-1, 4)
    assert np.array_equal(bits(part[s:e + 1]), bits(whole["accum"].reshape(-1, 4)[s:e + 1]))
    assert (part[:s] == 0).all() and (part[e + 1:] == 0).all()
    # empty range and zero passes are no-ops
    gpu.render_tile(rt.make_params(W, H, start=10, end=9, **kw))
    gpu.render_tile(rt.make_params(W, H, pass_count=0, **kw))
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).reshape(-1, 4)), bits(part))
    for bounce in (0, 1, 2):
        out, p = gpu_render(rt, gpu, sc, 64, 48, mode=rt.RT_MODE_PATH, max_bounce=bounce, antialias=0)
        o = port.render(sc.desc, p)
        assert np.array_equal(bits(out["accum"]), bits(o["accum"]))
    out, p = gpu_render(rt, gpu, sc, 1, 1, mode=rt.RT_MODE_PATH, max_bounce=4, antialias=1, seed=9)
    o = port.render(sc.desc, p)
    assert np.array_equal(bits(out["accum"]), bits(o["accum"]))


def test_error_behaviour(rt, gpu, data_dir):
    with pytest.raises(rt.RtError):
        gpu.render_tile(rt.make_params(8, 8, max_bounce=64))
    with pytest.raises(rt.RtError):
        gpu.render_tile(rt.make_params(8, 8, start=0, end=64))
    fresh = rt.GpuContext(0)
    with pytest.raises(rt.RtError):
        fresh.render_tile(rt.make_params(8, 8))           # no scene
    sc = rt.Scene([("sphere", (0, 0, 0), 1.0, ("diffuse", (1, 1, 1)))])
    fresh.upload_scene(sc)
    with pytest.raises(rt.RtError):
        fresh.render_tile(rt.make_params(8, 8))           # Diffuse without a unit-vector table
    # a node array that is not a pre-order binary tree is refused at upload (the walks rely on the nesting)
    sm = rt.Scene([("mesh", f"{data_dir}/TorusKnot.obj", ("diffuse", (1, 1, 1)))])
    mesh = sm.desc.contents.meshes[0]
    nodes, n = mesh.nodes, mesh.num_nodes
    inner = next(k for k in range(1, n) if nodes[k].tri < 0)
    leaf = next(k for k in range(1, n) if nodes[k].tri >= 0)
    for k, field, value in ((inner, "escape", inner + 1),            # inner node without children
                            (inner + 1, "escape", n),                # left subtree sticks out of its parent
                            (leaf, "escape", min(leaf + 2, n)),      # leaf with a subtree
                            (leaf, "tri", mesh.num_tris),            # leaf slot out of range
                            (0, "escape", n + 1)):                   # root escape past the array
        keep = getattr(nodes[k], field)
        setattr(nodes[k], field, value)
        try:
            if getattr(nodes[k], field) != keep:
                with pytest.raises(rt.RtError):
                    fresh.upload_scene(sm)
        finally:
            setattr(nodes[k], field, keep)
    fresh.upload_scene(sm)                                # intact again
    fresh.close()


# ---------------------------------------------------------------------------------------------------
# tier-1 primitive known-answer tests on the device functions
# ---------------------------------------------------------------------------------------------------
def _kat(rt, gpu, kind, rays, prims, width):
    import ctypes as C
    prims = np.ascontiguousarray(prims, np.float32).reshape(-1, width)
    n = len(prims)
    flags = np.zeros(n, np.int32)
    out7 = np.zeros((n, 7), np.float32)
    rp = None if rays is None else np.ascontiguousarray(rays, np.float32).ctypes.data
    rc = rt.load_library().rt_gpu_kat(gpu.handle, kind, rp, prims.ctypes.data, width, n, flags.ctypes.data, out7.ctypes.data)
    assert rc == 0
    return flags, out7


def test_kat_primitives_bit_exact(rt, gpu, port, ref):
    rng = np.random.default_rng(3)
    n = 100_000
    rays = random_rays(n, 11)
    # boxes around the scene incl. flat boxes (min == max on one axis, Appendix A3)
    lo = rng.normal(size=(n, 3)).astype(np.float32)
    ext = np.abs(rng.normal(size=(n, 3))).astype(np.float32)
    ext[: n // 8, 0] = 0.0
    boxes = np.concatenate([lo, lo + ext], 1)
    f, o = _kat(rt, gpu, 0, rays, boxes, 6)
    rf, rtmin = ref.kat_aabb(rays, boxes)
    np.testing.assert_array_equal(f, rf)
    np.testing.assert_array_equal(bits(o[:, 0]), bits(rtmin))
    tris = (rng.normal(size=(n, 9)) * 1.5).astype(np.float32)
    tris[: n // 10, 3:6] = tris[: n // 10, 0:3] + (rng.normal(size=(n // 10, 3)) * 1e-4).astype(np.float32)   # slivers: unnormalised normal (A7)
    for kind, prims, width, fn in ((1, tris, 9, ref.kat_triangle),
                                   (2, np.concatenate([rng.normal(size=(n, 3)), np.abs(rng.normal(size=(n, 1))) + 0.1], 1), 4, ref.kat_sphere),
                                   (3, np.concatenate([rng.normal(size=(n, 3)), rng.normal(size=(n, 3))], 1), 6, ref.kat_plane),
                                   (4, np.concatenate([rng.normal(size=(n, 6)), np.abs(rng.normal(size=(n, 1))) * 0.5 + 0.05], 1), 7, ref.kat_capsule)):
        prims = prims.astype(np.float32)
        f, o = _kat(rt, gpu, kind, rays, prims, width)
        rf, ro = fn(rays, prims)
        np.testing.assert_array_equal(f, rf)
        assert f.sum() > 100
        np.testing.assert_array_equal(bits(o), bits(ro))
    x = np.abs(rng.normal(size=n)).astype(np.float32) * np.float32(10) ** rng.integers(-6, 6, n).astype(np.float32)
    _, o = _kat(rt, gpu, 5, None, x, 1)
    np.testing.assert_array_equal(bits(o[:, 0]), bits(ref.kat_qrsqrt(x)))
    pabc = rng.normal(size=(n, 12)).astype(np.float32)
    _, o = _kat(rt, gpu, 6, None, pabc, 12)
    np.testing.assert_array_equal(bits(o[:, :3]), bits(ref.kat_barycentric(pabc)))
    rgb = rng.random(size=(n, 3)).astype(np.float32) * 1.2
    f, _ = _kat(rt, gpu, 7, None, rgb, 3)
    assert_display_close(f.view(np.uint32), ref.kat_display(rgb))


def test_kat_texture_sample_bit_exact(rt, gpu, ref, data_dir):
    spec = scenes.c3_unitychan(data_dir)
    sc = rt.Scene(spec)
    gpu.upload_scene(sc)
    rs = ref.build_scene(spec)
    rng = np.random.default_rng(5)
    uv = (rng.random(size=(50_000, 2)) * 3 - 1).astype(np.float32)
    uv[:100] = np.array([[0, 0], [1, 1], [0.5, 1.0], [1.0, 0.0]] * 25, np.float32)
    k = 0
    ntex = ref.mesh_counts(rs, 0)[4]
    for slot in range(ntex):
        if ref.mesh_texture(rs, 0, slot) is None:
            continue
        want = ref.kat_texture_sample(rs, 0, slot, uv)
        got = np.zeros((len(uv), 4), np.float32)
        rc = rt.load_library().rt_gpu_kat_texture(gpu.handle, k, uv.ctypes.data, len(uv), got.ctypes.data)
        assert rc == 0
        np.testing.assert_array_equal(bits(got), bits(want))
        k += 1
    assert k == 8
    ref.free_scene(rs)


# ---------------------------------------------------------------------------------------------------
# scheduling never changes results: pool overflow (retry passes), queue windows, refill thresholds
# ---------------------------------------------------------------------------------------------------
def test_pool_overflow_and_tuning_do_not_change_results(rt, port, data_dir):
    ctx = rt.GpuContext(0)
    sc = rt.Scene(scenes.default_scene(data_dir))       # ground plane: every camera ray becomes a path
    sc.set_unit_vectors(seed=2, count=1 << 18)
    ctx.upload_scene(sc)
    W, H = 320, 200
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=8, antialias=1, pass_count=2, seed=4)
    ref_img, ref_cnt = None, None
    for tune in ((32, 28, 8, 0), (32, 28, 8, 16), (64, 1, 0, 33), (128, 32, 16, 100), (32, 16, 4, 9)):
        ctx.set_tuning(*tune)       # pools of 16Ki / 33Ki / ... records against 512000 camera rays: many retry passes
        ctx.reset_accum(W, H)
        ctx.reset_counters()
        ctx.render_tile(p)
        img = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy()
        c = ctx.counters()
        if ref_img is None:
            ref_img, ref_cnt = img, c
            o = port.render(sc.desc, p, nthreads=8)
            frac, mean_err = stochastic_check(img, o["accum"])
            assert frac <= 2e-3 and mean_err <= 1e-3
            assert c["rays"] == o["counters"]["rays"] and c["camera_rays"] == W * H * 8
        else:
            assert np.array_equal(bits(img), bits(ref_img)), tune
            for k in ("rays", "camera_rays", "mesh_hits"):
                assert c[k] == ref_cnt[k], (tune, k)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("traverse", ["exact", "culled"])
def test_frontier_long_walks_are_bit_identical(rt, data_dir, traverse, monkeypatch):
    """The long-walk kernel (frontier expansion + leaf replay in slot order) against the lane-per-walk kernel:
    parking every walk after 8 / 40 node steps, or handing whole rounds to it, with 32-, 16- and 8-lane groups,
    changes neither a bit of the image nor — in exact mode — the visit counters (KdTree.cpp:128-195 order)."""
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    sc.set_unit_vectors(seed=5, count=1 << 18)
    W, H = 480, 270
    trav = rt.RT_TRAVERSE_EXACT if traverse == "exact" else rt.RT_TRAVERSE_CULLED
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=1, pass_count=2, seed=11, traverse=trav)
    ref_img, ref_cnt = None, None
    variants = [dict(RT_LONG_LIMIT="1000000", RT_SMALL_ROUND="0", RT_THIN_COUNT="0"),           # no walk ever parked
                dict(RT_LONG_LIMIT="8", RT_SMALL_ROUND="0", RT_THIN_COUNT="0", RT_LONG_GROUP_N="32"),
                dict(RT_LONG_LIMIT="40", RT_SMALL_ROUND="0", RT_THIN_COUNT="0", RT_LONG_GROUP_N="16"),
                dict(RT_LONG_LIMIT="8", RT_SMALL_ROUND="0", RT_THIN_COUNT="0", RT_LONG_GROUP_N="8"),
                dict(RT_LONG_LIMIT="2048", RT_SMALL_ROUND="100000000", RT_THIN_COUNT="0", RT_LONG_GROUP_N="32"),  # every round whole
                dict()]                                                                        # shipped defaults
    for env in variants:
        for k in ("RT_LONG_LIMIT", "RT_SMALL_ROUND", "RT_THIN_COUNT", "RT_THIN_LIMIT", "RT_LONG_GROUP_N"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ctx = rt.GpuContext(0)          # the knobs are read when a context is created
        ctx.upload_scene(sc)
        ctx.reset_accum(W, H)
        ctx.reset_counters()
        ctx.render_tile(p)
        img = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy()
        c = ctx.counters()
        ctx.close()
        if ref_img is None:
            ref_img, ref_cnt = img, c
            continue
        assert np.array_equal(bits(img), bits(ref_img)), env
        keys = ("rays", "camera_rays", "mesh_hits") + (("node_tests", "tri_tests") if traverse == "exact" else ())
        for k in keys:
            assert c[k] == ref_cnt[k], (env, k)


@pytest.mark.parametrize("traverse", ["exact", "culled"])
def test_packet_walk_is_bit_identical(rt, data_dir, traverse, monkeypatch):
    """Round 0 walked as 32-ray packets (rt_walk_packet_kernel) against the lane-per-walk kernel: no packets,
    (with and without the shared-memory stage for the top of the first mesh's tree, RT_TOP_STAGE),
    packets for round 0, packets for every round, packets that are always given up after their first window
    (every lane resumes lane by lane at its cursor), a probe window of 5 steps — same image bits, same ray and
    hit counts and, in exact mode, the reference's slab / triangle test counts.  Two meshes in the scene, so
    packets split into per-mesh groups."""
    spec = [("plane", (0.0, 1.0, 0.0), (0.0, -2.5, 0.0), ("checker", scenes.WHITE, 5.0)),
            ("mesh", f"{data_dir}/TorusKnot.obj", ("reflective", (0.9, 0.9, 0.9), 0.0)),
            ("mesh", f"{data_dir}/unitychan.obj", ("diffuse", scenes.WHITE))]
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=3, count=1 << 18)
    W, H = 512, 300
    trav = rt.RT_TRAVERSE_EXACT if traverse == "exact" else rt.RT_TRAVERSE_CULLED
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=6, antialias=1, pass_count=2, seed=21, traverse=trav)
    ref_img, ref_cnt = None, None
    knobs = ("RT_PACKET_ROUNDS", "RT_PACKET_MIN_LANES", "RT_PACKET_PROBE", "RT_TOP_STAGE", "RT_OCTO")
    variants = [dict(RT_PACKET_ROUNDS="0"),
                dict(RT_PACKET_ROUNDS="0", RT_OCTO="1"),           # every round of the culled traversal on the 8-wide tree
                dict(RT_OCTO="1"),
                dict(RT_PACKET_ROUNDS="0", RT_TOP_STAGE="1"),      # every round lane by lane, top of mesh 0's tree from shared memory
                dict(RT_TOP_STAGE="1"),
                dict(RT_PACKET_ROUNDS="1", RT_PACKET_MIN_LANES="0"),
                dict(RT_PACKET_ROUNDS="100", RT_PACKET_MIN_LANES="0"),
                dict(RT_PACKET_ROUNDS="100", RT_PACKET_MIN_LANES="33"),
                dict(RT_PACKET_ROUNDS="1", RT_PACKET_MIN_LANES="16", RT_PACKET_PROBE="5"),
                dict()]
    for env in variants:
        for k in knobs:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ctx = rt.GpuContext(0)          # the knobs are read when a context is created
        ctx.upload_scene(sc)
        ctx.reset_accum(W, H)
        ctx.reset_counters()
        ctx.render_tile(p)
        img = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy()
        c = ctx.counters()
        ctx.close()
        if ref_img is None:
            ref_img, ref_cnt = img, c
            continue
        assert same_bits(img, ref_img), env
        keys = ("rays", "camera_rays", "mesh_hits") + (("node_tests", "tri_tests") if traverse == "exact" else ())
        for k in keys:
            assert c[k] == ref_cnt[k], (env, k)


def test_push_owned_into_root_frame(rt, gpu, data_dir):
    """The peer-memory exchange: three 'ranks' (contexts of their own) write the tiles they own straight into
    the root context's accumulation buffer (rt_gpu_push_owned; here all on one device, so the root's frame is
    reachable by its plain device address) == the frame rendered by one context alone, bit for bit.  Odd frame
    size: clipped tiles at the right and bottom edges."""
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    sc.set_unit_vectors(seed=0, count=1 << 18)
    W, H, n = 333, 217, 3
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=6, antialias=1, seed=9, pass_count=2)
    full, _ = gpu_render(rt, gpu, sc, W, H, **kw)
    lib = rt.load_library()
    gpu.reset_accum(W, H)
    root_frame = lib.rt_gpu_accum_device_ptr(gpu.handle)
    p0 = rt.make_params(W, H, tile_size=32, tile_count=n, tile_rank=0, **kw)
    gpu.render_tile(p0)
    gpu.synchronize()
    for r in range(1, n):
        peer = rt.GpuContext(0)
        peer.upload_scene(sc)
        p = rt.make_params(W, H, tile_size=32, tile_count=n, tile_rank=r, **kw)
        peer.reset_accum(W, H)
        peer.render_tile(p)
        peer.push_owned(p, root_frame)
        peer.synchronize()
        peer.close()
    got = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert np.array_equal(bits(got), bits(full["accum"]))
    # a frame of another size is refused, and so is a null frame
    with pytest.raises(rt.RtError):
        gpu.push_owned(rt.make_params(W + 1, H, tile_size=32, tile_count=n, tile_rank=0, **kw), root_frame)


def test_frame_slots_and_host_delivery(rt, data_dir):
    """Two frames enqueued back to back on the two frame slots (they overlap on the device; their chunks rotate
    through the pipes) == the same frames rendered one after the other on one slot; and rt_gpu_deliver_owned:
    three 'ranks' write their own tiles of accuBuffer and bitcolor straight into ONE registered host frame ==
    the frame read back whole."""
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    sc.set_unit_vectors(seed=0, count=1 << 20)
    W, H = 640, 360
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=8, antialias=1, pass_count=4)
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)
    want = []
    for seed in (3, 4, 5):
        ctx.reset_accum(W, H)
        ctx.render_tile(rt.make_params(W, H, seed=seed, **kw))
        want.append((ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H), ctx.readback(rt.RT_READ_DISPLAY_ARGB8, W, H)))
    for k, seed in enumerate((3, 4, 5)):                    # no host synchronisation in between
        ctx.set_frame_slot(k & 1)
        ctx.reset_accum(W, H)
        ctx.render_tile(rt.make_params(W, H, seed=seed, **kw))
        if k == 1:
            ctx.set_frame_slot(0)                           # frame 0 is read while frame 1 is in flight
            assert np.array_equal(bits(ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(want[0][0]))
    ctx.set_frame_slot(1)
    assert np.array_equal(bits(ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(want[1][0]))
    ctx.set_frame_slot(0)
    assert np.array_equal(bits(ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(want[2][0]))
    np.testing.assert_array_equal(ctx.readback(rt.RT_READ_DISPLAY_ARGB8, W, H), want[2][1])
    with pytest.raises(rt.RtError):
        ctx.set_frame_slot(rt._abi.RT_GPU_FRAME_SLOTS)
    # delivery into a host frame: accuBuffer (16 B/px) followed by bitcolor (4 B/px), as bench.py lays it out
    npix = W * H
    host = np.zeros(npix * 20 + 64, np.uint8)          # + a header word for rt_gpu_signal_host
    dev = ctx.register_host_frame(host.ctypes.data, host.nbytes)
    n = 3
    for r in range(n):
        p = rt.make_params(W, H, seed=5, tile_size=32, tile_count=n, tile_rank=r, **kw)
        ctx.set_frame_slot(r & 1)
        ctx.reset_accum(W, H)
        ctx.render_tile(p)
        ctx.deliver_owned(p, dev, dev + npix * 16)
        ctx.signal_host(dev + npix * 20 + 4 * r, 100 + r)        # "rank r has delivered", ordered after the delivery
    for s in (0, 1):
        ctx.set_frame_slot(s)
        ctx.synchronize()
    assert np.array_equal(host[:npix * 16].view(np.uint32).reshape(H, W, 4), bits(want[2][0]))
    np.testing.assert_array_equal(host[npix * 16:npix * 20].view(np.uint32).reshape(H, W), want[2][1])
    np.testing.assert_array_equal(host[npix * 20:npix * 20 + 12].view(np.uint32), [100, 101, 102])
    ctx.unregister_host_frame(host.ctypes.data)
    ctx.close()


def test_device_pack_order_equals_host_tiles(rt, gpu, data_dir):
    """rt_gpu_pack_owned's dense layout == raytracerwin_b200.tiles.dense_index (what the gather relies on)."""
    import torch
    from raytracerwin_b200 import tiles
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    W, H, T, n = 333, 117, 32, 3
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=3, antialias=0)
    whole, _ = gpu_render(rt, gpu, sc, W, H, **kw)
    flat = whole["accum"].reshape(-1, 4)
    for r in range(n):
        p = rt.make_params(W, H, tile_size=T, tile_count=n, tile_rank=r, **kw)
        cnt = rt.owned_pixels(W, H, T, n, r)
        buf = torch.zeros((cnt, 4), dtype=torch.float32, device="cuda:0")
        gpu.pack_owned(p, buf.data_ptr(), buf.numel() * 4)
        gpu.synchronize()
        np.testing.assert_array_equal(bits(buf.cpu().numpy()), bits(flat[tiles.dense_index(W, H, T, n, r)]))
        with pytest.raises(rt.RtError):
            gpu.pack_owned(p, buf.data_ptr(), buf.numel() * 4 - 16)      # size-checked


# ---------------------------------------------------------------------------------------------------
# more scenes: several meshes, nothing at all, degenerate geometry, deep budgets, odd tilings
# ---------------------------------------------------------------------------------------------------
def test_two_meshes_and_analytic_shapes_between(rt, gpu, port, data_dir):
    """Two mesh shapes with a sphere between them in the shape list: one round per (segment x mesh),
    stale hit fields carried from mesh to sphere to mesh (Appendix A11)."""
    spec = [("mesh", f"{data_dir}/BlenderMonkey.obj", ("reflective", (0.9, 0.7, 0.5), 0.0)),
            ("sphere", (0.0, 0.0, 1.5), 0.45, ("combine", ("reflective", (0.6, 0.6, 0.9), 0.0), ("emissive", (0.1, 0.0, 0.0)))),
            ("plane", (0.0, 1.0, 0.0), (0.0, -2.0, 0.0), ("checker", (1, 1, 1), 5.0)),
            ("mesh", f"{data_dir}/TorusKnot.obj", ("blend", ("reflective", (1, 1, 1), 0.0), ("diffuse", (0.3, 0.8, 0.4)), 0.5))]
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=8, count=1 << 18)
    W, H = 400, 300
    for mode, kw in ((rt.RT_MODE_PRIMARY, {}), (rt.RT_MODE_WHITTED, dict(antialias=0)), (rt.RT_MODE_PREVIEW, dict(antialias=1, seed=1)),
                     (rt.RT_MODE_PATH, dict(max_bounce=7, antialias=1, pass_count=2, seed=6))):
        out, p = gpu_render(rt, gpu, sc, W, H, mode=mode, **kw)
        p.traverse = rt.RT_TRAVERSE_EXACT
        o = port.render(sc.desc, p, nthreads=8, want_primary=(mode == rt.RT_MODE_PRIMARY))
        if mode == rt.RT_MODE_PRIMARY:
            np.testing.assert_array_equal(out["ids"], o["ids"])
            np.testing.assert_array_equal(bits(out["dist"]), bits(o["dist"]))
        else:
            key = "preview" if mode == rt.RT_MODE_PREVIEW else "accum"
            assert same_bits(out[key], o[key]), mode
            assert out["counters"]["rays"] == o["counters"]["rays"]


def test_empty_and_sky_only_scenes(rt, gpu, port):
    sc = rt.Scene([])
    W, H = 64, 40
    out, p = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PATH, max_bounce=3, antialias=1, pass_count=2, seed=1)
    o = port.render(sc.desc, p)
    assert np.array_equal(bits(out["accum"]), bits(o["accum"]))
    assert out["counters"]["rays"] == W * H * 8 == out["counters"]["camera_rays"]
    out, p = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PRIMARY)
    assert (out["ids"] == -1).all() and (out["dist"] == 0).all()


def test_degenerate_triangles_and_nan_rays(rt, gpu, port):
    """Zero-area and sliver triangles (NaN barycentrics, Appendix A9), an unnormalised tiny normal (A7), and rays
    with zero / NaN / infinite components: identical to the restatement, NaNs included."""
    pts = np.array([[-1, -1, 0], [1, -1, 0], [0, 1, 0],            # a proper triangle
                    [0.5, 0.5, 0.5], [0.5, 0.5, 0.5], [0.5, 0.5, 0.5],   # a point
                    [-2, 0, 1], [2, 0, 1], [0, 1e-5, 1],           # a sliver (|cross|^2 < FLT_EPSILON)
                    [-1, -1, -1], [1, -1, -1], [3, -1, -1]], np.float32)   # collinear
    idx = np.arange(12, dtype=np.int32).reshape(4, 3)
    sc = rt.Scene()
    sc.add_mesh_arrays(pts, idx, material=("reflective", (0.8, 0.8, 0.8), 0.0))
    gpu.upload_scene(sc)
    rays = random_rays(50_000, 3, scale=2.0)
    rays[:8, 3:6] = 0.0                                                # zero direction: every slab disabled
    rays[8:16, 3] = np.nan
    rays[16:24, 0] = np.inf
    rays[24:32, 6] = 0.0                                               # zero length
    ps, pt, ph = port.trace_rays(sc.desc, rays)
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        gs, gt, gh = gpu.trace_rays(rays, tr)
        np.testing.assert_array_equal(gs, ps)
        np.testing.assert_array_equal(gt, pt)
        np.testing.assert_array_equal(bits(gh), bits(ph))
    W, H = 200, 150
    out, p = gpu_render(rt, gpu, sc, W, H, mode=rt.RT_MODE_PATH, max_bounce=4, antialias=0)
    o = port.render(sc.desc, p)
    assert same_bits(out["accum"], o["accum"])


def test_deep_budget_odd_tiles_pass_offsets(rt, gpu, port, data_dir):
    sc = rt.Scene(scenes.c2_monkey(data_dir))
    W, H = 211, 97
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=32, antialias=1, seed=9)
    out, p = gpu_render(rt, gpu, sc, W, H, pass_begin=5, pass_count=3, **kw)
    o = port.render(sc.desc, p, nthreads=8)
    assert np.array_equal(bits(out["accum"]), bits(o["accum"]))
    # 5 ranks, 8-pixel tiles, more ranks than some rows of tiles; assembled frame == the single frame
    acc = np.zeros((H, W, 4), np.float32)
    for r in range(5):
        gpu.reset_accum(W, H)
        gpu.render_tile(rt.make_params(W, H, pass_begin=5, pass_count=3, tile_size=8, tile_count=5, tile_rank=r, **kw))
        part = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
        assert not ((acc[..., 3] > 0) & (part[..., 3] > 0)).any()
        acc += part
    assert np.array_equal(bits(acc), bits(out["accum"]))


def test_headless_program_run(rt, tmp_path, data_dir):
    """RayTracerProgram::Run: preview pass, N accumulation passes, PNG of the display buffer."""
    import ctypes as C
    sc = rt.Scene()
    sc.setup_default_scene(data_dir)
    sc.set_unit_vectors(seed=1, count=1 << 18)
    png = str(tmp_path / "out.png")
    secs, rays = C.c_double(), C.c_uint64()
    rc = rt.load_library().rt_host_program_run(sc._h, 0, 160, 120, 3, 10, 4, png.encode(), C.byref(secs), C.byref(rays))
    assert rc == 0, rt.load_library().rt_host_last_error()
    assert rays.value > 160 * 120 * 12 and secs.value > 0
    wh = (C.c_int32 * 2)()
    ch = C.c_int32()
    px = C.POINTER(C.c_uint8)()
    assert rt.load_library().rt_host_decode_png(png.encode(), wh, C.byref(ch), C.byref(px)) == 0
    assert (wh[0], wh[1], ch.value) == (160, 120, 3)
    img = np.ctypeslib.as_array(px, (120, 160, 3)).copy()
    rt.load_library().rt_host_free(px)
    assert img.std() > 10            # an actual picture
