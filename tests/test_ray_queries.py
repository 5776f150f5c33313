"""Ray queries on device memory (rt_gpu_query_rays, GpuContext.query_rays): batches of the caller's rays through the
wavefront kernels, nearest hit and occlusion, results in torch tensors on the stream that made the rays.

Every result is held to an existing pin: the nearest hit to the restatement's find_intersection and to the test hook
rt_gpu_trace_rays (both bit for bit), occlusion to the restatement's shadow query (flags and, in exact mode, the
slab / triangle test counts)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import scenes
from conftest import ROOT, bits, same_bits

TRAVERSALS = (0, 1)         # RT_TRAVERSE_EXACT, RT_TRAVERSE_CULLED


def random_rays(n, seed, scale=3.0):
    """Incoherent rays from everywhere (inside boxes, behind, short), with axis-aligned and zero-component directions."""
    rng = np.random.default_rng(seed)
    o = rng.normal(size=(n, 3)).astype(np.float32) * np.float32(scale)
    tgt = rng.normal(size=(n, 3)).astype(np.float32) * np.float32(0.8)
    d = tgt - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    dist = rng.choice(np.array([1000.0, 10.0, 3.0, 0.5], np.float32), size=n)
    rays = np.concatenate([o, d.astype(np.float32), dist[:, None]], 1).astype(np.float32)
    k = n // 16
    rays[:k, 3:6] = 0.0
    rays[:k, 3 + (np.arange(k) % 3)] = np.where(rng.random(k) < 0.5, -1.0, 1.0)
    rays[k:2 * k, 4] = 0.0
    nrm = np.linalg.norm(rays[k:2 * k, 3:6], axis=1, keepdims=True)
    rays[k:2 * k, 3:6] /= np.where(nrm == 0, 1, nrm)
    return rays


def pinhole_rays(W, H, block_order, eye=(0.0, 0.0, 7.0), dir_z=-0.5, dist=1000.0):
    """The reference's camera (RayTracerProgram.cpp:133-165, no jitter) for a W x H frame, in row order or in the
    8x4-pixel blocks of the render's work list (32 consecutive rays = one block)."""
    if block_order:
        assert W % 8 == 0 and H % 4 == 0
        lane = np.arange(32)
        bx, by = np.meshgrid(np.arange(W // 8), np.arange(H // 4))
        x = (bx.reshape(-1, 1) * 8 + (lane & 7)).reshape(-1)
        y = (by.reshape(-1, 1) * 4 + (lane >> 3)).reshape(-1)
    else:
        y, x = np.divmod(np.arange(W * H), W)
    aspect = np.float32(W) / np.float32(H)
    dx = -(x - W // 2).astype(np.float32) / np.float32(W * 2) * aspect
    dy = -(y - H // 2).astype(np.float32) / np.float32(H * 2)
    d = np.stack([dx, dy, np.full_like(dx, dir_z)], 1).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = np.broadcast_to(np.asarray(eye, np.float32), d.shape)
    return np.concatenate([o, d, np.full((len(d), 1), dist, np.float32)], 1).astype(np.float32)


def bounce_rays(hit, n, seed):
    """Bounce-like rays from primary hit points: off the surface along the normal, into its hemisphere."""
    rng = np.random.default_rng(seed)
    h = hit[hit[:, 6] > 0]
    h = h[rng.integers(0, len(h), n)]
    nrm = h[:, 3:6]
    u = rng.normal(size=(n, 3)).astype(np.float32)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    d = nrm + u
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), np.float32(1e-6))
    o = h[:, 0:3] + nrm * np.float32(1e-4)
    return np.concatenate([o, d, np.full((n, 1), 1000.0, np.float32)], 1).astype(np.float32)


# The restatement's shadow query, occluded() of oracle/rt_oracle.c (the function the Whitted tests pin to the
# reference's CalculateLightColor, RayTracerScene.cpp:152-164), on arbitrary rays.  It is static there, so this
# wrapper includes the restatement whole and is compiled with its flags for the session.
OCCLUDED_SRC = r"""
#include "rt_oracle.c"
/* flags[k] = 1 when an accepted hit lies within ray k's Distance; counters = rays, shadow_rays, node_tests,
 * tri_tests, mesh_walks */
int occluded_rays(const rt_scene_desc* sc, const float* rays, int n, int32_t* flags, uint64_t* counters)
{
    cnt_t c; memset(&c, 0, sizeof c);
    for (int k = 0; k < n; k++) {
        const float* q = rays + 7 * (size_t)k;
        ray_t r = { V(q[0], q[1], q[2]), V(q[3], q[4], q[5]), q[6] };
        flags[k] = occluded(sc, &r, &c);
    }
    counters[0] = c.rays; counters[1] = c.shadow_rays; counters[2] = c.node_tests;
    counters[3] = c.tri_tests; counters[4] = c.mesh_walks;
    return 0;
}
"""


@pytest.fixture(scope="session")
def occluded_rays(tmp_path_factory):
    """occluded_rays(desc, rays) -> (int32 flags, {rays, shadow_rays, node_tests, tri_tests, mesh_walks})"""
    d = tmp_path_factory.mktemp("occluded")
    src, lib = d / "occluded.c", d / "liboccluded.so"
    src.write_text(OCCLUDED_SRC)
    subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                    "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"),
                    "-o", str(lib), str(src), "-lm", "-lpthread"], check=True)
    L = C.CDLL(str(lib))
    L.occluded_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]

    def run(desc, rays):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        flags = np.zeros(len(rays), np.int32)
        cnt = np.zeros(5, np.uint64)
        L.occluded_rays(C.cast(desc, C.c_void_p), rays.ctypes.data, len(rays), flags.ctypes.data, cnt.ctypes.data)
        return flags, dict(zip(("rays", "shadow_rays", "node_tests", "tri_tests", "mesh_walks"), map(int, cnt)))
    return run


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def query(gpu, rays, traverse, any_hit=False):
    """GpuContext.query_rays on host rays, results back as numpy (the copy waits for the query's stream)."""
    out = gpu.query_rays(to_dev(rays), any_hit=any_hit, traverse=traverse)
    if any_hit:
        return out.cpu().numpy()
    return out["shape"].cpu().numpy(), out["tri"].cpu().numpy(), out["hit"].cpu().numpy()


def assert_same_nearest(got, want):
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1], want[1])
    assert same_bits(got[2], want[2])


# ---------------------------------------------------------------------------------------------------
# layout of the query struct (no GPU)
# ---------------------------------------------------------------------------------------------------
def test_ray_query_layout_matches_c(rt):
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "rt_gpu.h"
int main(void) {
  printf("size %zu\n", sizeof(rt_ray_query));
  printf("rays %zu\n", offsetof(rt_ray_query, rays)); printf("n %zu\n", offsetof(rt_ray_query, n));
  printf("kind %zu\n", offsetof(rt_ray_query, kind)); printf("traverse %zu\n", offsetof(rt_ray_query, traverse));
  printf("shape %zu\n", offsetof(rt_ray_query, shape)); printf("tri %zu\n", offsetof(rt_ray_query, tri));
  printf("hit %zu\n", offsetof(rt_ray_query, hit));
  printf("nearest %d\n", RT_QUERY_NEAREST); printf("any %d\n", RT_QUERY_ANY);
  return 0; }
'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "q.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "q")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    q = rt._abi.rt_ray_query
    assert C.sizeof(q) == out["size"]
    for f in ("rays", "n", "kind", "traverse", "shape", "tri", "hit"):
        assert getattr(q, f).offset == out[f], f
    assert (rt.RT_QUERY_NEAREST, rt.RT_QUERY_ANY) == (out["nearest"], out["any"])


def test_occlusion_restatement_agrees_with_nearest(rt, port, occluded_rays, data_dir):
    """The shadow loop accepts a ray iff the nearest-hit loop finds a shape: the first shape to accept sees the ray's
    full Distance in both.  Exact-mode test counts: every slab and triangle test of the loop up to that shape."""
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    rays = random_rays(20_000, 13)
    flags, cnt = occluded_rays(sc.desc, rays)
    shape, _, _ = port.trace_rays(sc.desc, rays)
    np.testing.assert_array_equal(flags, (shape >= 0).astype(np.int32))
    assert cnt["rays"] == cnt["shadow_rays"] == len(rays)
    assert 0 < flags.mean() < 1 and cnt["node_tests"] > 0 and cnt["tri_tests"] > 0 and cnt["mesh_walks"] > 0


# ---------------------------------------------------------------------------------------------------
# nearest hit and occlusion against the restatement and the hook
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["default_scene", "deterministic_mix", "c3_unitychan"])
def test_nearest_and_any_bit_exact(rt, gpu, port, occluded_rays, data_dir, scene_name):
    sc = rt.Scene(getattr(scenes, scene_name)(data_dir))
    gpu.upload_scene(sc)
    rays = random_rays(200_000, 7)
    want = port.trace_rays(sc.desc, rays)
    flags, pcnt = occluded_rays(sc.desc, rays)
    assert (want[0] >= 0).mean() > 0.05
    # the first shape to accept a ray sees its full Distance in both loops: occluded == nearest hit exists
    np.testing.assert_array_equal(flags, (want[0] >= 0).astype(np.int32))
    for tr in TRAVERSALS:
        assert_same_nearest(query(gpu, rays, tr), want)
        assert_same_nearest(query(gpu, rays, tr), gpu.trace_rays(rays, tr))
        gpu.synchronize()
        gpu.reset_counters()
        gpu.synchronize()
        np.testing.assert_array_equal(query(gpu, rays, tr, any_hit=True), flags)
        c = gpu.counters()
        assert c["rays"] == c["shadow_rays"] == len(rays) and c["camera_rays"] == 0
        if tr == 0:
            for k in ("node_tests", "tri_tests", "mesh_walks"):
                assert c[k] == pcnt[k], k


@pytest.mark.gpu
def test_counters_equal_the_hook(rt, gpu, data_dir):
    """Exact mode: one nearest-hit batch adds what the hook adds on the same rays."""
    sc = rt.Scene(scenes.default_scene(data_dir))
    gpu.upload_scene(sc)
    rays = random_rays(200_000, 5)
    counts = []
    for run in (lambda: query(gpu, rays, 0), lambda: gpu.trace_rays(rays, 0)):
        gpu.reset_counters()
        gpu.synchronize()
        run()
        counts.append(gpu.counters())
    for k in ("rays", "node_tests", "tri_tests", "mesh_walks", "mesh_hits", "shadow_rays", "camera_rays"):
        assert counts[0][k] == counts[1][k], k
    assert counts[0]["camera_rays"] == 0 and counts[0]["rays"] == len(rays) and counts[0]["mesh_walks"] > 0


@pytest.mark.gpu
def test_large_coherent_and_shuffled_batches(rt, gpu, data_dir):
    """Pinhole rays in 8x4-block and in row order (round-0 packets), the same rays shuffled (packets given up,
    walked lane by lane) and bounce-like rays from the primary hits, 2 M each, against the hook."""
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    gpu.upload_scene(sc)
    W, H = 1920, 1080
    blocks = pinhole_rays(W, H, True)
    rows = pinhole_rays(W, H, False)
    shuffled = blocks[np.random.default_rng(1).permutation(len(blocks))]
    want_blocks = gpu.trace_rays(blocks, 1)
    assert (want_blocks[0] >= 0).mean() > 0.01
    bounce = bounce_rays(want_blocks[2], 2_000_000, 2)
    for name, rays in (("blocks", blocks), ("rows", rows), ("shuffled", shuffled), ("bounce", bounce)):
        want = want_blocks if name == "blocks" else gpu.trace_rays(rays, 1)
        got = query(gpu, rays, 1)
        assert_same_nearest(got, want)
        np.testing.assert_array_equal(query(gpu, rays, 1, any_hit=True), (want[0] >= 0).astype(np.int32))
    assert_same_nearest(query(gpu, blocks, 0), gpu.trace_rays(blocks, 0))


@pytest.mark.gpu
def test_rounds_empty_and_degenerate_scenes(rt, gpu, port, occluded_rays, data_dir):
    """Two meshes with analytic shapes between them (several rounds, stale hit fields carried across shapes), an
    empty scene, and degenerate triangles with zero / NaN / infinite / zero-length rays."""
    two = [("mesh", f"{data_dir}/BlenderMonkey.obj", ("reflective", (0.9, 0.7, 0.5), 0.0)),
           ("sphere", (0.0, 0.0, 1.5), 0.45, ("combine", ("reflective", (0.6, 0.6, 0.9), 0.0), ("emissive", (0.1, 0.0, 0.0)))),
           ("plane", (0.0, 1.0, 0.0), (0.0, -2.0, 0.0), ("checker", (1, 1, 1), 5.0)),
           ("mesh", f"{data_dir}/TorusKnot.obj", ("blend", ("reflective", (1, 1, 1), 0.0), ("diffuse", (0.3, 0.8, 0.4)), 0.5))]
    pts = np.array([[-1, -1, 0], [1, -1, 0], [0, 1, 0],
                    [0.5, 0.5, 0.5], [0.5, 0.5, 0.5], [0.5, 0.5, 0.5],
                    [-2, 0, 1], [2, 0, 1], [0, 1e-5, 1],
                    [-1, -1, -1], [1, -1, -1], [3, -1, -1]], np.float32)
    degenerate = rt.Scene()
    degenerate.add_mesh_arrays(pts, np.arange(12, dtype=np.int32).reshape(4, 3), material=("reflective", (0.8, 0.8, 0.8), 0.0))
    weird = random_rays(50_000, 3, scale=2.0)
    weird[:8, 3:6] = 0.0
    weird[8:16, 3] = np.nan
    weird[16:24, 0] = np.inf
    weird[24:32, 6] = 0.0
    for sc, rays in ((rt.Scene(two), random_rays(200_000, 9)), (rt.Scene([]), random_rays(10_000, 4)), (degenerate, weird)):
        gpu.upload_scene(sc)
        want = port.trace_rays(sc.desc, rays)
        flags, _ = occluded_rays(sc.desc, rays)
        for tr in TRAVERSALS:
            assert_same_nearest(query(gpu, rays, tr), want)
            np.testing.assert_array_equal(query(gpu, rays, tr, any_hit=True), flags)


@pytest.mark.gpu
def test_batch_sizes_and_small_pools(rt, gpu, data_dir):
    sc = rt.Scene(scenes.default_scene(data_dir))
    gpu.upload_scene(sc)
    for n in (0, 1, 31, 33, (1 << 20) + 7):
        rays = random_rays(n, 100 + n) if n else np.zeros((0, 7), np.float32)
        got = query(gpu, rays, 1)
        assert got[0].shape == (n,) and got[2].shape == (n, 11)
        if n:
            assert_same_nearest(got, gpu.trace_rays(rays, 1))
            np.testing.assert_array_equal(query(gpu, rays, 1, any_hit=True), (got[0] >= 0).astype(np.int32))
    # pools of 16 Ki records: the batch runs in many pieces over all pipes, with the same results
    ctx = rt.GpuContext(0)
    ctx.set_tuning(pool_kpaths=16)
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    ctx.upload_scene(sc)
    rays = np.concatenate([pinhole_rays(640, 360, True), random_rays(100_000, 8)])
    for tr in TRAVERSALS:
        assert_same_nearest(query(ctx, rays, tr), ctx.trace_rays(rays, tr))
    ctx.close()


# ---------------------------------------------------------------------------------------------------
# streams: ordered on the caller's stream, invisible to renders
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_query_on_a_side_stream_without_host_sync(rt, gpu, data_dir):
    import torch
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    gpu.upload_scene(sc)
    rays = pinhole_rays(640, 360, True)
    want = gpu.trace_rays(rays, 1)
    dev = torch.device("cuda", 0)
    src = to_dev(rays)
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        made = torch.empty_like(src)
        torch.cuda._sleep(20_000_000)               # the rays are late: a query not ordered after them reads garbage
        made.copy_(src)
        out = gpu.query_rays(made)
        occ = gpu.query_rays(made, any_hit=True)
        shape = out["shape"].clone()                 # consumed on the same stream, no host synchronisation
        hit = out["hit"] * 1.0
        tri = out["tri"] + 0
        occ = occ.clone()
    s.synchronize()
    np.testing.assert_array_equal(shape.cpu().numpy(), want[0])
    np.testing.assert_array_equal(tri.cpu().numpy(), want[1])
    assert same_bits(hit.cpu().numpy(), want[2])
    np.testing.assert_array_equal(occ.cpu().numpy(), (want[0] >= 0).astype(np.int32))


@pytest.mark.gpu
def test_queries_between_render_calls_change_nothing(rt, data_dir):
    """Frames on slots 0 and 1 with query batches enqueued between the calls == the same frames without them
    (accuBuffer bits; counters less what the queries add)."""
    import torch
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    sc.set_unit_vectors(seed=0, count=1 << 18)
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
            if with_queries:
                results.append(ctx.query_rays(rays))
            ctx.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=6, antialias=1, pass_count=2, seed=seed))
            if with_queries:
                results.append(ctx.query_rays(rays, any_hit=True))
        imgs = []
        for s in (0, 1):
            ctx.set_frame_slot(s)
            imgs.append(ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy())
        torch.cuda.synchronize()
        return imgs, ctx.counters(), results

    imgs0, c0, _ = frames(False)
    imgs1, c1, results = frames(True)
    for a, b in zip(imgs0, imgs1):
        assert np.array_equal(bits(a), bits(b))
    ctx.set_frame_slot(0)
    ctx.reset_counters()
    ctx.synchronize()
    for _ in range(2):
        ctx.query_rays(rays)
        ctx.query_rays(rays, any_hit=True)
    torch.cuda.synchronize()
    cq = ctx.counters()
    for k in keys:
        assert c1[k] == c0[k] + cq[k], k
    want = ctx.trace_rays(rays.cpu().numpy(), 1)
    for r in results[0::2]:
        np.testing.assert_array_equal(r["shape"].cpu().numpy(), want[0])
    for r in results[1::2]:
        np.testing.assert_array_equal(r.cpu().numpy(), (want[0] >= 0).astype(np.int32))
    ctx.close()


# ---------------------------------------------------------------------------------------------------
# errors leave the context usable
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_inputs_are_rejected(rt, data_dir):
    import torch
    abi = rt._abi
    lib = rt.load_library()
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    rays = random_rays(4_000, 12)
    dev_rays = to_dev(rays)
    ctx = rt.GpuContext(0)
    with pytest.raises(rt.RtError):
        ctx.query_rays(dev_rays)                    # before upload_scene
    ctx.upload_scene(sc)
    want = ctx.trace_rays(rays, 1)

    def usable():
        assert_same_nearest(query(ctx, rays, 1), want)

    bad = [rays, dev_rays.cpu(), dev_rays.double(), dev_rays[:, :6].contiguous(), dev_rays.t().contiguous().t(),
           dev_rays[::2], dev_rays.reshape(-1)]
    if torch.cuda.device_count() > 1:
        bad.append(dev_rays.to("cuda:1"))
    for b in bad:
        with pytest.raises((rt.RtError, ValueError)):
            ctx.query_rays(b)
        usable()
    for kw in (dict(want_tri=True), dict(want_hit=True)):
        with pytest.raises(rt.RtError):
            ctx.query_rays(dev_rays, any_hit=True, **kw)
        usable()
    # the C ABI itself
    n = len(rays)
    shape = torch.empty(n, dtype=torch.int32, device="cuda:0")
    tri = torch.empty(n, dtype=torch.int32, device="cuda:0")
    host_shape = np.zeros(n, np.int32)

    def call(**kw):
        f = dict(rays=dev_rays.data_ptr(), n=n, kind=abi.RT_QUERY_NEAREST, traverse=abi.RT_TRAVERSE_CULLED,
                 shape=shape.data_ptr(), tri=None, hit=None)
        f.update(kw)
        q = abi.rt_ray_query(f["rays"], f["n"], f["kind"], f["traverse"], f["shape"], f["tri"], f["hit"])
        rc = lib.rt_gpu_query_rays(ctx.handle, C.byref(q), None)
        ctx.synchronize()
        return rc

    assert call() == abi.RT_OK
    np.testing.assert_array_equal(shape.cpu().numpy(), want[0])
    assert call(n=0, rays=None, shape=None) == abi.RT_OK
    for kw in (dict(n=-1), dict(kind=2), dict(traverse=2), dict(rays=None), dict(shape=None),
               dict(kind=abi.RT_QUERY_ANY, tri=tri.data_ptr()), dict(rays=rays.ctypes.data), dict(shape=host_shape.ctypes.data)):
        assert call(**kw) == abi.RT_ERR_INVALID, kw
        assert lib.rt_gpu_last_error(ctx.handle)
        usable()
    assert lib.rt_gpu_query_rays(ctx.handle, None, None) == abi.RT_ERR_INVALID
    ctx.close()
