"""Radiance queries on device memory (rt_gpu_radiance_rays, GpuContext.radiance_rays): RayTrace's path, its preview
colour and the Whitted composition of the caller's rays, through the render's wavefront kernels.

Every result is held to an existing pin: the restatement's ray_trace / whitted (oracle/rt_oracle.c, pinned to the
reference by the render tests) on the same rays and RNG streams, bit for bit with its ray and test counts, and
render_tile itself, GPU against GPU, when the rays are the render's camera rays."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import scenes
from conftest import ROOT, same_bits
from test_ray_queries import bounce_rays, pinhole_rays, random_rays, to_dev

TRAVERSALS = (0, 1)         # RT_TRAVERSE_EXACT, RT_TRAVERSE_CULLED
PATH, PREVIEW, WHITTED = 0, 1, 2
TOL = 1e-4

# The restatement's RayTrace and Whitted composition on arbitrary rays with caller-chosen RNG streams, and its camera
# (the rays render_tile shoots).  Both are static there, so this wrapper includes the restatement whole and is
# compiled with its flags for the session.
RADIANCE_SRC = r"""
#include "rt_oracle.c"
/* rgb[k] = ray_trace / whitted of ray k, drawing from {rt_rng_key(seed, streams[k], sample), first_draw};
 * counters = rays, camera_rays, shadow_rays, node_tests, tri_tests, mesh_walks */
int radiance_rays(const rt_scene_desc* sc, const float* rays, int n, int mode, int max_bounce, uint32_t seed,
                  uint32_t sample, const uint32_t* streams, uint32_t first_draw, float* rgb, uint64_t* counters)
{
    cnt_t c; memset(&c, 0, sizeof c);
    for (int k = 0; k < n; k++) {
        const float* q = rays + 7 * (size_t)k;
        ray_t r = { V(q[0], q[1], q[2]), V(q[3], q[4], q[5]), q[6] };
        rng_t rng = { rt_rng_key(seed, streams[k], sample), first_draw };
        v3 L = mode == RT_MODE_WHITTED ? whitted(sc, &r, &c) : ray_trace(sc, &r, max_bounce, mode == RT_MODE_PREVIEW, &rng, &c);
        rgb[3 * (size_t)k] = L.x; rgb[3 * (size_t)k + 1] = L.y; rgb[3 * (size_t)k + 2] = L.z;
    }
    counters[0] = c.rays; counters[1] = c.camera_rays; counters[2] = c.shadow_rays;
    counters[3] = c.node_tests; counters[4] = c.tri_tests; counters[5] = c.mesh_walks;
    return 0;
}
/* the camera ray of pixels[k] for pass p->pass_begin (sub = -1: un-jittered, else sub-sample sub of an antialiased
 * pass), and the RNG position after it */
int camera_rays(const rt_scene_desc* sc, const rt_render_params* p, const int32_t* pixels, int n, int sub,
                float* rays, uint32_t* draws)
{
    for (int k = 0; k < n; k++) {
        uint32_t sample = sub >= 0 ? (uint32_t)(p->pass_begin * 4 + sub) : (uint32_t)p->pass_begin;
        rng_t rng = { rt_rng_key(p->seed, (uint32_t)pixels[k], sample), 0 };
        ray_t r = camera_ray(sc, p, pixels[k], sub, &rng);
        float* o = rays + 7 * (size_t)k;
        o[0] = r.o.x; o[1] = r.o.y; o[2] = r.o.z; o[3] = r.d.x; o[4] = r.d.y; o[5] = r.d.z; o[6] = r.dist;
        draws[k] = rng.n;
    }
    return 0;
}
"""

COUNTERS = ("rays", "camera_rays", "shadow_rays", "node_tests", "tri_tests", "mesh_walks")


class Restatement:
    def __init__(self, lib):
        self.L = lib

    def radiance_rays(self, desc, rays, mode, max_bounce, seed, sample, streams, first_draw):
        """-> (float32 rgb (N, 3), {rays, camera_rays, shadow_rays, node_tests, tri_tests, mesh_walks})"""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        streams = np.ascontiguousarray(streams, np.uint32).reshape(-1)
        assert len(streams) == len(rays)
        rgb = np.zeros((len(rays), 3), np.float32)
        cnt = np.zeros(6, np.uint64)
        self.L.radiance_rays(C.cast(desc, C.c_void_p), rays.ctypes.data, len(rays), mode, max_bounce, seed, sample,
                             streams.ctypes.data, first_draw, rgb.ctypes.data, cnt.ctypes.data)
        return rgb, dict(zip(COUNTERS, map(int, cnt)))

    def camera_rays(self, desc, params, pixels, sub):
        """-> (float32 rays (N, 7), uint32 RNG position after each ray)"""
        pixels = np.ascontiguousarray(pixels, np.int32)
        rays = np.zeros((len(pixels), 7), np.float32)
        draws = np.zeros(len(pixels), np.uint32)
        self.L.camera_rays(C.cast(desc, C.c_void_p), C.byref(params), pixels.ctypes.data, len(pixels), sub,
                           rays.ctypes.data, draws.ctypes.data)
        return rays, draws


@pytest.fixture(scope="session")
def restatement(tmp_path_factory):
    d = tmp_path_factory.mktemp("radiance")
    src, lib = d / "radiance.c", d / "libradiance.so"
    src.write_text(RADIANCE_SRC)
    subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                    "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"),
                    "-o", str(lib), str(src), "-lm", "-lpthread"], check=True)
    L = C.CDLL(str(lib))
    L.radiance_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    L.camera_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return Restatement(L)


def radiance(ctx, rays, **kw):
    """GpuContext.radiance_rays on host rays (and a host rng_stream), result back as numpy (N, 4)."""
    import torch
    if kw.get("rng_stream") is not None:
        kw["rng_stream"] = to_dev(np.ascontiguousarray(kw["rng_stream"], np.uint32).view(np.int32))
    out = ctx.radiance_rays(to_dev(np.ascontiguousarray(rays, np.float32)), **kw)
    assert out.dtype == torch.float32 and tuple(out.shape) == (len(rays), 4)
    return out.cpu().numpy()


def counted(ctx, fn):
    """(result of fn(), the counters it added)"""
    ctx.synchronize()
    ctx.reset_counters()
    ctx.synchronize()
    r = fn()
    ctx.synchronize()
    return r, ctx.counters()


def scene_of(rt, name, data_dir):
    sc = rt.Scene(getattr(scenes, name)(data_dir))
    sc.set_unit_vectors(seed=0, count=1 << 18)
    return sc


def batches(ctx, seed):
    """pinhole (8x4-block order), incoherent (axis-aligned and zero-component directions included) and bounce-like
    rays off the hits of both"""
    pin = pinhole_rays(192, 128, True)
    rnd = random_rays(24_000, seed)
    hits = np.concatenate([ctx.trace_rays(pin, 1)[2], ctx.trace_rays(rnd, 1)[2]])
    out = dict(pinhole=pin, random=rnd)
    if (hits[:, 6] > 0).any():
        out["bounce"] = bounce_rays(hits, 24_000, seed + 1)
    return out


# ---------------------------------------------------------------------------------------------------
# layout of the query struct (no GPU)
# ---------------------------------------------------------------------------------------------------
def test_radiance_query_layout_matches_c(rt):
    fields = ("rays", "n", "mode", "max_bounce", "traverse", "seed", "sample", "rng_stream", "rng_stream_base",
              "first_draw", "rgba")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rt_gpu.h\"\nint main(void) {\n"
    src += '  printf("size %zu\\n", sizeof(rt_radiance_query));\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_radiance_query, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "q.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "q")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    q = rt._abi.rt_radiance_query
    assert C.sizeof(q) == out["size"]
    for f in fields:
        assert getattr(q, f).offset == out[f], f
    assert "rt_gpu_radiance_rays" in rt._abi.GPU_PROTOTYPES


# ---------------------------------------------------------------------------------------------------
# against the restatement, bit for bit
# ---------------------------------------------------------------------------------------------------
MODES = ((PATH, 1), (PATH, 4), (PATH, 10), (PREVIEW, 10), (WHITTED, 10))


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["c1_torusknot", "c2_monkey", "c2_monkey_null", "deterministic_mix", "c3_unitychan"])
def test_bit_exact_vs_restatement(rt, gpu, restatement, data_dir, scene_name):
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    for k, (name, rays) in enumerate(batches(gpu, 21).items()):
        n = len(rays)
        base, seed, sample, first = 1000 * k + 5, 7 + k, 3, 2 * (k % 2)
        for mode, bounce in MODES:
            want, wc = restatement.radiance_rays(sc.desc, rays, mode, bounce, seed, sample,
                                                 base + np.arange(n, dtype=np.uint32), first)
            for tr in TRAVERSALS:
                got, c = counted(gpu, lambda: radiance(gpu, rays, mode=mode, max_bounce=bounce, seed=seed, sample=sample,
                                                       rng_stream_base=base, first_draw=first, traverse=tr))
                where = (scene_name, name, mode, bounce, tr)
                assert same_bits(got[:, :3], want), where
                assert not got[:, 3].any(), where
                assert c["rays"] == wc["rays"] and c["shadow_rays"] == wc["shadow_rays"], where
                assert c["camera_rays"] == 0, where
                if tr == 0:
                    assert c["node_tests"] == wc["node_tests"] and c["tri_tests"] == wc["tri_tests"], where
                    assert c["mesh_walks"] == wc["mesh_walks"], where
            if mode == WHITTED:
                assert wc["shadow_rays"] > 0
            if mode == PATH and bounce == 10 and scene_name in ("c2_monkey", "deterministic_mix"):
                assert wc["rays"] > n          # paths did bounce


@pytest.mark.gpu
def test_default_scene_within_the_render_bar(rt, gpu, restatement, data_dir):
    """Fuzzy reflection calls sinf / cosf / acosf, whose CUDA and glibc results differ in the last ulp and can steer a
    path elsewhere: the render's bar per ray, >= 99.8 % within 1e-4 and the mean within 0.1 %."""
    sc = scene_of(rt, "default_scene", data_dir)
    gpu.upload_scene(sc)
    for k, (name, rays) in enumerate(batches(gpu, 31).items()):
        streams = np.random.default_rng(k).integers(0, 1 << 32, len(rays), dtype=np.uint64).astype(np.uint32)
        for mode, bounce in MODES:
            want, _ = restatement.radiance_rays(sc.desc, rays, mode, bounce, 11, 0, streams, 0)
            got = radiance(gpu, rays, mode=mode, max_bounce=bounce, seed=11, sample=0, rng_stream=streams)[:, :3]
            bad = (np.abs(got - want) > TOL).any(1) | (np.isnan(got) != np.isnan(want)).any(1)
            assert bad.mean() <= 2e-3, (name, mode, bounce, bad.mean())
            ok = np.isfinite(got).all(1) & np.isfinite(want).all(1)
            assert abs(got[ok].mean() - want[ok].mean()) <= 1e-3 * want[ok].mean(), (name, mode, bounce)


@pytest.mark.gpu
def test_negative_distance_is_not_culled(rt, gpu, port, data_dir):
    """A bounce after a hit beyond the segment's end (a capsule hit, which is not compared with Distance, or a triangle
    hit of a ray with |d| > 1) has a negative Distance, and the reference then accepts triangles behind the origin.
    The culled traversal must not skip them: nearest-hit queries of such rays equal the restatement in both
    traversals."""
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    rays = random_rays(100_000, 61, scale=1.0)
    rays[::2, 6] *= np.float32(-0.01)
    want = port.trace_rays(sc.desc, rays)
    assert (want[0][::2] >= 0).mean() > 0.01
    for tr in TRAVERSALS:
        got = gpu.query_rays(to_dev(rays), traverse=tr)
        np.testing.assert_array_equal(got["shape"].cpu().numpy(), want[0])
        np.testing.assert_array_equal(got["tri"].cpu().numpy(), want[1])
        assert same_bits(got["hit"].cpu().numpy(), want[2])


# ---------------------------------------------------------------------------------------------------
# the render's own camera rays give the render, GPU against GPU
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["c3_unitychan", "default_scene"])
def test_equals_render_tile(rt, gpu, restatement, data_dir, scene_name):
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    W, H = 160, 120
    pixels = np.arange(W * H, dtype=np.int32)
    zero = np.float32(0.0)
    for p, seed in ((0, 3), (5, 9)):
        # one un-jittered pass after a reset: accum = 0 + RayTrace(camera ray)
        params = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, antialias=0, pass_begin=p, pass_count=1, seed=seed)
        gpu.reset_accum(W, H)
        gpu.render_tile(params)
        acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).reshape(-1, 4)
        cam, draws = restatement.camera_rays(sc.desc, params, pixels, -1)
        assert not draws.any()
        got = radiance(gpu, cam, mode=PATH, max_bounce=10, seed=seed, sample=p, rng_stream=pixels)
        assert same_bits(zero + got[:, :3], acc[:, :3]), (scene_name, p)
        # four jittered rays per pixel: sample 4p + i, two draws spent on the jitter; the pass colour folded as
        # ThreadWorker_Render folds it, then AddPixel on a reset buffer
        params.antialias = 1
        gpu.reset_accum(W, H)
        gpu.render_tile(params)
        acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).reshape(-1, 4)
        col = np.zeros((W * H, 3), np.float32)
        for i in range(4):
            cam, draws = restatement.camera_rays(sc.desc, params, pixels, i)
            assert (draws == 2).all()
            col = col + radiance(gpu, cam, mode=PATH, max_bounce=10, seed=seed, sample=4 * p + i, rng_stream=pixels,
                                 first_draw=2)[:, :3]
        col = col / np.float32(4.0)
        assert same_bits(zero + col, acc[:, :3]), (scene_name, p)
        # the preview pass: RT_READ_PREVIEW_RGBA_F32 holds the pass colour itself
        params.mode = rt.RT_MODE_PREVIEW
        gpu.reset_accum(W, H)
        gpu.render_tile(params)
        prev = gpu.readback(rt.RT_READ_PREVIEW_RGBA_F32, W, H).reshape(-1, 4)
        col = np.zeros((W * H, 3), np.float32)
        for i in range(4):
            cam, _ = restatement.camera_rays(sc.desc, params, pixels, i)
            col = col + radiance(gpu, cam, mode=PREVIEW, max_bounce=10, seed=seed, sample=4 * p + i, rng_stream=pixels,
                                 first_draw=2)[:, :3]
        assert same_bits(col / np.float32(4.0), prev[:, :3]), (scene_name, p)


@pytest.mark.gpu
def test_whitted_equals_render_tile(rt, gpu, restatement, data_dir):
    sc = scene_of(rt, "c1_torusknot", data_dir)
    gpu.upload_scene(sc)
    W, H = 320, 240
    pixels = np.arange(W * H, dtype=np.int32)
    params = rt.make_params(W, H, mode=rt.RT_MODE_WHITTED, antialias=0, pass_count=1)
    gpu.reset_accum(W, H)
    gpu.render_tile(params)
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).reshape(-1, 4)
    cam, _ = restatement.camera_rays(sc.desc, params, pixels, -1)
    for tr in TRAVERSALS:
        got = radiance(gpu, cam, mode=WHITTED, rng_stream=pixels, traverse=tr)
        assert same_bits(np.float32(0.0) + got[:, :3], acc[:, :3])
    assert (acc[:, :3].sum(1) == 0).any() and (acc[:, :3].sum(1) > 0).any()


# ---------------------------------------------------------------------------------------------------
# scheduling never changes a bit
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_invariance(rt, gpu, data_dir):
    import torch
    sc = scene_of(rt, "default_scene", data_dir)
    gpu.upload_scene(sc)
    pin = pinhole_rays(256, 128, True)
    rays = np.concatenate([pin, random_rays(40_000, 41), bounce_rays(gpu.trace_rays(pin, 1)[2], 20_000, 42)])
    n = len(rays)
    base = 777
    kw = dict(mode=PATH, max_bounce=10, seed=5, sample=2)
    want = radiance(gpu, rays, rng_stream_base=base, **kw)
    assert (want[:, :3] > 0).any()
    # exact traversal; explicit stream ids; a shuffled batch with its stream ids shuffled alike
    assert same_bits(radiance(gpu, rays, rng_stream_base=base, traverse=0, **kw), want)
    streams = (base + np.arange(n)).astype(np.uint32)
    assert same_bits(radiance(gpu, rays, rng_stream=streams, **kw), want)
    perm = np.random.default_rng(3).permutation(n)
    assert same_bits(radiance(gpu, rays[perm], rng_stream=streams[perm], **kw), want[perm])
    # batches of 1, 31, 33 rays anywhere in the batch (implicit ids: the base moves with them)
    for size, at in ((1, 0), (1, 4321), (31, 0), (33, 1000), (33, n - 33)):
        got = radiance(gpu, rays[at:at + size], rng_stream_base=base + at, **kw)
        assert same_bits(got, want[at:at + size]), (size, at)
    # pools of 16 Ki records (the batch runs in many pieces) on four pipes and on one
    ctx = rt.GpuContext(0)
    ctx.set_tuning(pool_kpaths=16)
    ctx.upload_scene(sc)
    for pipes in (4, 1):
        ctx.set_pipes(pipes)
        assert same_bits(radiance(ctx, rays, rng_stream_base=base, **kw), want), pipes
        assert same_bits(radiance(ctx, rays, rng_stream=streams, traverse=0, **kw), want), pipes
    ctx.close()
    # a batch of 100 003 rays, WHITTED and PREVIEW too: in one piece and in many
    big = np.concatenate([rays, random_rays(100_003 - n, 43)])
    ctx = rt.GpuContext(0)
    ctx.set_tuning(pool_kpaths=16)
    ctx.upload_scene(sc)
    for mode in (PATH, PREVIEW, WHITTED):
        one = radiance(gpu, big, mode=mode, max_bounce=10, seed=1, rng_stream_base=9)
        assert same_bits(radiance(ctx, big, mode=mode, max_bounce=10, seed=1, rng_stream_base=9), one), mode
        assert same_bits(one[:n], radiance(gpu, rays, mode=mode, max_bounce=10, seed=1, rng_stream_base=9)), mode
    ctx.close()
    # a side stream, no host synchronisation: ordered after the rays are made, consumed on the same stream
    dev = torch.device("cuda", 0)
    src = to_dev(rays)
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        made = torch.empty_like(src)
        torch.cuda._sleep(20_000_000)               # the rays are late: a query not ordered after them reads garbage
        made.copy_(src)
        out = torch.full((n, 4), -1.0, dtype=torch.float32, device=dev)
        r = gpu.radiance_rays(made, rng_stream_base=base, out=out, **kw)
        assert r is out
        res = out * 1.0
    s.synchronize()
    assert same_bits(res.cpu().numpy(), want)


# ---------------------------------------------------------------------------------------------------
# edges
# ---------------------------------------------------------------------------------------------------
def sky(d):
    """RayTrace's miss colour (RayTracerScene.cpp:92-93), one rounding per operation"""
    t = np.float32(0.5) * (d[:, 1] + np.float32(1.0))
    one_t = np.float32(1.0) - t
    return np.stack([np.float32(1.0) * one_t + np.float32(c) * t for c in (0.5, 0.7, 1.0)], 1).astype(np.float32)


@pytest.mark.gpu
def test_edges(rt, gpu, restatement, data_dir):
    sc = scene_of(rt, "deterministic_mix", data_dir)
    gpu.upload_scene(sc)
    rays = random_rays(20_000, 51)
    # max_bounce 0: RayTrace(ray, 0) is black, and nothing is traced
    for mode in (PATH, PREVIEW):
        got, c = counted(gpu, lambda: radiance(gpu, rays, mode=mode, max_bounce=0))
        assert not got.any() and not np.signbit(got).any()
        assert c["rays"] == 0
    # an empty scene: the sky, in every mode
    empty = rt.Scene([])
    gpu.upload_scene(empty)
    for mode in (PATH, PREVIEW, WHITTED):
        got = radiance(gpu, rays, mode=mode, max_bounce=3)
        want, _ = restatement.radiance_rays(empty.desc, rays, mode, 3, 0, 0, np.arange(len(rays)), 0)
        assert same_bits(got[:, :3], want)
        assert same_bits(want, sky(rays[:, 3:6]))
    # analytic shapes only: no mesh to walk, yet paths bounce for as many rounds as the budget allows
    analytic = rt.Scene([s for s in scenes.deterministic_mix(data_dir) if s[0] != "mesh"])
    gpu.upload_scene(analytic)
    for mode, bounce in MODES:
        want, wc = restatement.radiance_rays(analytic.desc, rays, mode, bounce, 4, 1, 50 + np.arange(len(rays)), 0)
        got, c = counted(gpu, lambda: radiance(gpu, rays, mode=mode, max_bounce=bounce, seed=4, sample=1, rng_stream_base=50))
        assert same_bits(got[:, :3], want), (mode, bounce)
        assert c["rays"] == wc["rays"] and c["shadow_rays"] == wc["shadow_rays"]
        if mode == PATH and bounce == 10:
            assert wc["rays"] > len(rays)


@pytest.mark.gpu
def test_radiance_between_render_calls_changes_nothing(rt, data_dir):
    """Frames on slots 0 and 1 with radiance batches enqueued between the calls == the same frames without them
    (accumulation and display buffers, preview buffer, frame slot; counters less what the batches add)."""
    import torch
    sc = scene_of(rt, "c3_unitychan", data_dir)
    W, H = 320, 200
    rays = to_dev(np.concatenate([pinhole_rays(320, 200, True), random_rays(50_000, 6)]))
    keys = ("rays", "camera_rays", "shadow_rays", "mesh_hits", "mesh_walks")
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)

    def frames(with_queries):
        results = []
        for s in (0, 1):
            ctx.set_frame_slot(s)
            ctx.synchronize()
        ctx.set_frame_slot(0)
        ctx.reset_counters()
        ctx.synchronize()
        for s, seed in ((0, 3), (1, 4)):
            ctx.set_frame_slot(s)
            ctx.reset_accum(W, H)
            ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PREVIEW, antialias=1, pass_count=1, seed=seed))
            if with_queries:
                results.append(ctx.radiance_rays(rays, max_bounce=6, seed=seed))
            ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=6, antialias=1, pass_count=2, seed=seed))
            if with_queries:
                results.append(ctx.radiance_rays(rays, mode=WHITTED))
                assert ctx._lib.rt_gpu_get_frame_slot(ctx.handle) == s
        out = []
        for s in (0, 1):
            ctx.set_frame_slot(s)
            out.append([ctx.readback(w, W, H).copy() for w in (rt.RT_READ_ACCUM_RGBN_F32, rt.RT_READ_DISPLAY_ARGB8,
                                                                rt.RT_READ_PREVIEW_RGBA_F32)])
        torch.cuda.synchronize()
        return out, ctx.counters(), results

    imgs0, c0, _ = frames(False)
    imgs1, c1, results = frames(True)
    for a, b in zip(imgs0, imgs1):
        for x, y in zip(a, b):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    ctx.set_frame_slot(0)
    ctx.reset_counters()
    ctx.synchronize()
    for seed in (3, 4):
        ctx.radiance_rays(rays, max_bounce=6, seed=seed)
        ctx.radiance_rays(rays, mode=WHITTED)
    torch.cuda.synchronize()
    cq = ctx.counters()
    for k in keys:
        assert c1[k] == c0[k] + cq[k], k
    assert cq["camera_rays"] == 0 and cq["shadow_rays"] > 0
    for r, seed in zip(results[0::2], (3, 4)):
        assert same_bits(r.cpu().numpy(), radiance(ctx, rays.cpu().numpy(), max_bounce=6, seed=seed))
    ctx.close()


# ---------------------------------------------------------------------------------------------------
# errors leave the context usable
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_inputs_are_rejected(rt, data_dir):
    import torch
    abi = rt._abi
    lib = rt.load_library()
    sc = scene_of(rt, "deterministic_mix", data_dir)
    rays = random_rays(4_000, 12)
    dev_rays = to_dev(rays)
    ctx = rt.GpuContext(0)
    n = len(rays)
    rgba = torch.empty((n + 1, 4), dtype=torch.float32, device="cuda:0")
    streams = torch.arange(n, dtype=torch.int32, device="cuda:0")

    def call(**kw):
        f = dict(rays=dev_rays.data_ptr(), n=n, mode=abi.RT_MODE_PATH, max_bounce=4, traverse=abi.RT_TRAVERSE_CULLED,
                 seed=0, sample=0, rng_stream=None, rng_stream_base=0, first_draw=0, rgba=rgba.data_ptr())
        f.update(kw)
        q = abi.rt_radiance_query(*[f[k] for k, _ in abi.rt_radiance_query._fields_])
        rc = lib.rt_gpu_radiance_rays(ctx.handle, C.byref(q), None)
        ctx.synchronize()
        return rc

    with pytest.raises(rt.RtError):
        ctx.radiance_rays(dev_rays)                 # before upload_scene
    assert call() == abi.RT_ERR_NO_SCENE
    assert lib.rt_gpu_last_error(ctx.handle)
    ctx.upload_scene(sc)
    want = radiance(ctx, rays, max_bounce=4)

    def usable():
        assert same_bits(radiance(ctx, rays, max_bounce=4), want)

    assert call() == abi.RT_OK
    assert same_bits(rgba[:n].cpu().numpy(), want)
    assert call(rng_stream=streams.data_ptr()) == abi.RT_OK
    assert same_bits(rgba[:n].cpu().numpy(), want)
    assert call(n=0, rays=None, rgba=None) == abi.RT_OK
    host_rgba = np.zeros((n, 4), np.float32)
    host_streams = np.zeros(n, np.uint32)
    for kw in (dict(n=-1), dict(mode=abi.RT_MODE_PRIMARY), dict(mode=4), dict(mode=-1), dict(max_bounce=-1),
               dict(max_bounce=33), dict(traverse=2), dict(rays=None), dict(rgba=None),
               dict(rays=rays.ctypes.data), dict(rgba=host_rgba.ctypes.data), dict(rng_stream=host_streams.ctypes.data),
               dict(rgba=rgba.data_ptr() + 4)):
        assert call(**kw) == abi.RT_ERR_INVALID, kw
        assert lib.rt_gpu_last_error(ctx.handle)
        usable()
    assert lib.rt_gpu_radiance_rays(ctx.handle, None, None) == abi.RT_ERR_INVALID
    # 52 meshes x 10 segments: more walks per path than the round table holds (as render_tile counts them)
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    many = rt.Scene()
    for k in range(52):
        many.add_mesh_arrays(tri + np.float32(k), np.arange(3, dtype=np.int32).reshape(1, 3), material=("reflective", (0.5, 0.5, 0.5), 0.0))
    ctx.upload_scene(many)
    assert call(max_bounce=10) == abi.RT_ERR_INVALID
    assert "round table" in lib.rt_gpu_last_error(ctx.handle).decode()
    assert call(max_bounce=9) == abi.RT_OK
    ctx.upload_scene(sc)
    usable()
    # the torch wrapper
    bad = [rays, dev_rays.cpu(), dev_rays.double(), dev_rays[:, :6].contiguous(), dev_rays.t().contiguous().t(),
           dev_rays[::2], dev_rays.reshape(-1)]
    for b in bad:
        with pytest.raises((rt.RtError, ValueError)):
            ctx.radiance_rays(b)
        usable()
    for kw in (dict(rng_stream=streams.cpu()), dict(rng_stream=streams.long()), dict(rng_stream=streams[:-1]),
               dict(rng_stream=torch.arange(2 * n, dtype=torch.int32, device="cuda:0")[::2]),
               dict(out=rgba[:n].cpu()), dict(out=rgba[:n].double()), dict(out=rgba), dict(out=rgba[:n, :3]),
               dict(out=rgba.t().contiguous().t()[:n]), dict(mode=rt.RT_MODE_PRIMARY), dict(max_bounce=-1)):
        with pytest.raises((rt.RtError, ValueError)):
            ctx.radiance_rays(dev_rays, **kw)
        usable()
    ctx.close()
