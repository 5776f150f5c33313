"""Movable cameras (rt_gpu_render_view, GpuContext.render_tile(params, camera), rt.look_at / rt.camera): the render of
render_tile from a camera of the call's own.

Every result is held to an existing pin: render_tile itself (no camera, or the identity basis with the scene's own eye,
dir_z and distance, bit for bit), and the restatement (oracle/rt_oracle.c, pinned to the reference by the render tests)
with its camera ray given the basis rule of include/rt_gpu.h: its ray_trace / whitted / find_intersection over those
rays, bit for bit with its ray and test counts."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import scenes
from conftest import ROOT, bits, same_bits
from test_ray_queries import to_dev

PATH, PREVIEW, WHITTED, PRIMARY = 0, 1, 2, 3
EXACT, CULLED = 0, 1

# The restatement's camera_ray with the camera of rt_gpu_render_view, and its render_pixel over those rays.  Its
# functions are static, so this wrapper includes the restatement whole and is compiled with its flags for the session.
VIEW_SRC = r"""
#include "rt_oracle.c"
static int identity_basis(const rt_camera* cam)
{
    for (int c = 0; c < 3; c++)
        if (cam->right[c] != (c == 0 ? 1.0f : 0.0f) || cam->up[c] != (c == 1 ? 1.0f : 0.0f) || cam->back[c] != (c == 2 ? 1.0f : 0.0f))
            return 0;
    return 1;
}

/* camera_ray with v = (dx + ox, dy + oy, dir_z) taken into the world by the camera's basis */
static ray_t view_ray(const rt_render_params* p, const rt_camera* cam, int pixel, int sub, rng_t* rng)
{
    float dx, dy;
    pixel_base(p, pixel, &dx, &dy);
    float ox = 0.0f, oy = 0.0f;
    if (sub >= 0) {
        const float inv_pixel_radius = 1.0f / (p->width * 4);
        const float offset_radius = inv_pixel_radius * 0.5f;
        ox = (sub & 1) ? inv_pixel_radius : 0.0f;
        oy = (sub & 2) ? inv_pixel_radius : 0.0f;
        ox += (rng_random(rng) - 0.5f) * offset_radius;
        oy += (rng_random(rng) - 0.5f) * offset_radius;
    }
    v3 v = V(dx + ox, dy + oy, cam->dir_z);
    if (!identity_basis(cam)) {
        float w[3];
        for (int c = 0; c < 3; c++) w[c] = (v.x * cam->right[c] + v.y * cam->up[c]) + v.z * cam->back[c];
        v = V(w[0], w[1], w[2]);
    }
    ray_t r = { ld3(cam->eye), normalized(v), cam->ray_distance };
    return r;
}

/* the camera ray of pixels[k] for pass p->pass_begin (sub = -1: un-jittered, else sub-sample sub), and the RNG
 * position after it */
int view_rays(const rt_render_params* p, const rt_camera* cam, const int32_t* pixels, int n, int sub, float* rays, uint32_t* draws)
{
    for (int k = 0; k < n; k++) {
        uint32_t sample = sub >= 0 ? (uint32_t)(p->pass_begin * 4 + sub) : (uint32_t)p->pass_begin;
        rng_t rng = { rt_rng_key(p->seed, (uint32_t)pixels[k], sample), 0 };
        ray_t r = view_ray(p, cam, pixels[k], sub, &rng);
        float* o = rays + 7 * (size_t)k;
        o[0] = r.o.x; o[1] = r.o.y; o[2] = r.o.z; o[3] = r.d.x; o[4] = r.d.y; o[5] = r.d.z; o[6] = r.dist;
        draws[k] = rng.n;
    }
    return 0;
}

/* render_pixel of the restatement with view_ray for camera_ray, over every owned pixel of [start, end] (one thread):
 * accum is ADDED to; preview / ids / pdist as rt_oracle_render_ex writes them.
 * counters = rays, camera_rays, shadow_rays, node_tests, tri_tests, mesh_walks */
int render_view(const rt_scene_desc* sc, const rt_render_params* p, const rt_camera* cam, int first_row, int last_row,
                float* accum, int32_t* ids, float* pdist, float* preview, uint64_t* counters)
{
    cnt_t c; memset(&c, 0, sizeof c);
    for (int pixel = p->start; pixel <= p->end; pixel++) {
        if (pixel / p->width < first_row || pixel / p->width > last_row || !owns_pixel(p, pixel)) continue;
        if (p->mode == RT_MODE_PRIMARY) {
            rng_t rng = { 0, 0 };
            ray_t r = view_ray(p, cam, pixel, -1, &rng);
            hit_t h = { {0,0,0}, {0,0,0}, 0.0f, {1.0f, 1.0f, 1.0f}, 1.0f };
            int tri = -1;
            c.camera_rays++;
            int shape = find_intersection(sc, r, &h, &tri, &c);
            ids[2 * (size_t)pixel] = shape; ids[2 * (size_t)pixel + 1] = shape >= 0 ? tri : -1;
            pdist[pixel] = shape >= 0 ? h.dist : 0.0f;
            continue;
        }
        float* a = accum + 4 * (size_t)pixel;
        v3 sum = V(a[0], a[1], a[2]);
        int num = (int)a[3];
        v3 last = V(0, 0, 0);
        for (int pass = p->pass_begin; pass < p->pass_begin + p->pass_count; pass++) {
            v3 col = V(0, 0, 0);
            if (p->antialias) {
                for (int i = 0; i < 4; i++) {
                    rng_t rng = { rt_rng_key(p->seed, (uint32_t)pixel, (uint32_t)(pass * 4 + i)), 0 };
                    ray_t r = view_ray(p, cam, pixel, i, &rng);
                    c.camera_rays++;
                    v3 s = p->mode == RT_MODE_WHITTED ? whitted(sc, &r, &c)
                                                      : ray_trace(sc, &r, p->max_bounce, p->mode == RT_MODE_PREVIEW, &rng, &c);
                    col = add(col, s);
                }
                col = V(col.x / 4.0f, col.y / 4.0f, col.z / 4.0f);
            } else {
                rng_t rng = { rt_rng_key(p->seed, (uint32_t)pixel, (uint32_t)pass), 0 };
                ray_t r = view_ray(p, cam, pixel, -1, &rng);
                c.camera_rays++;
                col = p->mode == RT_MODE_WHITTED ? whitted(sc, &r, &c)
                                                 : ray_trace(sc, &r, p->max_bounce, p->mode == RT_MODE_PREVIEW, &rng, &c);
            }
            sum = add(sum, col); num++;
            last = col;
        }
        if (p->mode == RT_MODE_PREVIEW) {
            float* q = preview + 4 * (size_t)pixel; q[0] = last.x; q[1] = last.y; q[2] = last.z; q[3] = 1.0f;
            continue;
        }
        a[0] = sum.x; a[1] = sum.y; a[2] = sum.z; a[3] = (float)num;
    }
    counters[0] = c.rays; counters[1] = c.camera_rays; counters[2] = c.shadow_rays;
    counters[3] = c.node_tests; counters[4] = c.tri_tests; counters[5] = c.mesh_walks;
    return 0;
}
"""

COUNTERS = ("rays", "camera_rays", "shadow_rays", "node_tests", "tri_tests", "mesh_walks")


class ViewRestatement:
    def __init__(self, lib):
        self.L = lib

    def view_rays(self, params, cam, pixels, sub):
        """-> (float32 rays (N, 7), uint32 RNG position after each ray)"""
        pixels = np.ascontiguousarray(pixels, np.int32)
        rays = np.zeros((len(pixels), 7), np.float32)
        draws = np.zeros(len(pixels), np.uint32)
        self.L.view_rays(C.byref(params), C.byref(cam), pixels.ctypes.data, len(pixels), sub, rays.ctypes.data,
                         draws.ctypes.data)
        return rays, draws

    def render(self, desc, params, cam):
        """-> dict(accum, preview (H, W, 4), ids (H, W, 2), dist (H, W), counters) of one call on fresh buffers,
        rows split over threads as the restatement's own render splits them"""
        from concurrent.futures import ThreadPoolExecutor
        W, H = params.width, params.height
        accum = np.zeros((H, W, 4), np.float32)
        preview = np.zeros((H, W, 4), np.float32)
        ids = np.full((H, W, 2), -1, np.int32)
        dist = np.zeros((H, W), np.float32)
        step = 8
        rows = [(r, min(r + step, H) - 1) for r in range(0, H, step)]
        cnts = [np.zeros(6, np.uint64) for _ in rows]

        def run(k):
            self.L.render_view(C.cast(desc, C.c_void_p), C.byref(params), C.byref(cam), rows[k][0], rows[k][1],
                               accum.ctypes.data, ids.ctypes.data, dist.ctypes.data, preview.ctypes.data,
                               cnts[k].ctypes.data)

        with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
            list(ex.map(run, range(len(rows))))
        total = sum(cnts)
        return dict(accum=accum, preview=preview, ids=ids, dist=dist, counters=dict(zip(COUNTERS, map(int, total))))


@pytest.fixture(scope="session")
def view_restatement(tmp_path_factory):
    d = tmp_path_factory.mktemp("camera")
    src, lib = d / "view.c", d / "libview.so"
    src.write_text(VIEW_SRC)
    subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                    "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"),
                    "-o", str(lib), str(src), "-lm", "-lpthread"], check=True)
    L = C.CDLL(str(lib))
    L.view_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.render_view.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_void_p]
    return ViewRestatement(L)


def scene_of(rt, name, data_dir):
    sc = rt.Scene(getattr(scenes, name)(data_dir))
    sc.set_unit_vectors(seed=0, count=1 << 18)
    return sc


def mesh_box(sc):
    """(center, half extent) of the union of the scene's mesh bounds"""
    d = sc.desc.contents
    lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
    for i in range(d.num_shapes):
        s = d.shapes[i]
        if s.type == 3:                                     # RT_SHAPE_MESH
            lo = np.minimum(lo, list(s.bounds_min))
            hi = np.maximum(hi, list(s.bounds_max))
    return (lo + hi) / 2, (hi - lo) / 2


def cameras(rt, sc):
    """the cameras every scene is rendered from: name -> rt_camera"""
    c, h = mesh_box(sc)
    r = float(np.linalg.norm(h)) * 1.3 + 0.2
    a = 2.0
    return {
        # identity basis: the reference's generator from another eye, image plane and distance
        "translated": rt.camera(c + np.array([0.4, 0.3, r]), (1, 0, 0), (0, 1, 0), (0, 0, 1), dir_z=-0.7, ray_distance=60.0),
        "orbit": rt.look_at(c + r * np.array([math.sin(a), 0.35, math.cos(a)]), c),
        "steep_up": rt.look_at(c + np.array([0.0, 0.2 * r, 0.6 * r]), c + np.array([0.0, 4.0 * r, 0.3 * r])),
        "steep_down": rt.look_at(c + np.array([0.2, 1.5 * r, 0.3 * r]), c + np.array([0.0, -2.0 * r, 0.0])),
        "inside_mesh": rt.look_at(c, c + np.array([1.0, 0.2, -0.3])),
        "below_plane": rt.look_at((0.3, -3.0, 1.5 * r), (0.0, -1.0, 0.0)),
        # a quarter turn about y: exact zeros, yet not the identity
        "zero_components": rt.camera(c + np.array([r, 0.0, 0.0]), (0, 0, -1), (0, 1, 0), (1, 0, 0), dir_z=-0.5),
        "non_orthonormal": rt.camera(c + np.array([0.5, 0.4, r]), (1.2, 0.1, 0.0), (0.2, 0.9, 0.1), (0.1, -0.2, 1.1),
                                     dir_z=-0.6, ray_distance=500.0),
    }


def render(rt, ctx, params, cam, reads=None):
    """one call on freshly reset buffers and counters -> dict of readbacks and counters"""
    W, H = params.width, params.height
    ctx.reset_accum(W, H)
    ctx.synchronize()
    ctx.reset_counters()
    ctx.synchronize()
    if cam is False:
        ctx.render_tile(params)
    elif cam is None:
        assert ctx._lib.rt_gpu_render_view(ctx.handle, C.byref(params), None) == 0
    else:
        ctx.render_tile(params, cam)
    ctx.synchronize()
    return read_all(rt, ctx, W, H, reads, preview=params.mode == PREVIEW)


def read_all(rt, ctx, W, H, reads=None, preview=False):
    """the frame buffers (the preview buffer exists once a preview pass has been rendered) and the counters"""
    if reads is None:
        reads = dict(accum=rt.RT_READ_ACCUM_RGBN_F32, display=rt.RT_READ_DISPLAY_ARGB8, ids=rt.RT_READ_PRIMARY_IDS_I32X2,
                     dist=rt.RT_READ_PRIMARY_DIST_F32)
        if preview:
            reads["preview"] = rt.RT_READ_PREVIEW_RGBA_F32
    out = {k: ctx.readback(w, W, H).copy() for k, w in reads.items()}
    out["counters"] = ctx.counters()
    return out


# the counters that do not depend on scheduling (node_visits / tri_visits of the culled walk depend on how walks are
# parked and resumed)
KEYS = ("rays", "camera_rays", "shadow_rays", "node_tests", "tri_tests", "mesh_hits", "mesh_walks")


def same_frame(a, b):
    """-> the first readback or counter in which a and b differ, or None"""
    for k in a:
        if k == "counters":
            for c in KEYS:
                if a[k][c] != b[k][c]:
                    return f"counter {c}: {a[k][c]} != {b[k][c]}"
        elif not np.array_equal(np.ascontiguousarray(a[k]).view(np.uint8), np.ascontiguousarray(b[k]).view(np.uint8)):
            return k
    return None


# ---------------------------------------------------------------------------------------------------
# no GPU: layout, declaration, look_at
# ---------------------------------------------------------------------------------------------------
def test_camera_layout_matches_c(rt):
    fields = ("eye", "right", "up", "back", "dir_z", "ray_distance")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rt_gpu.h\"\nint main(void) {\n"
    src += '  printf("size %zu\\n", sizeof(rt_camera));\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_camera, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "q.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "q")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    cam = rt._abi.rt_camera
    assert C.sizeof(cam) == out["size"] == 56
    for f in fields:
        assert getattr(cam, f).offset == out[f], f


def test_render_view_is_declared_and_exported(rt):
    header = open(os.path.join(ROOT, "include", "rt_gpu.h")).read()
    assert "int rt_gpu_render_view(rt_gpu_ctx* ctx, const rt_render_params* params, const rt_camera* camera);" in header
    assert "rt_gpu_render_view" in rt._abi.GPU_PROTOTYPES
    lib = rt.load_library()
    assert lib.rt_gpu_render_view.argtypes[2] is C.POINTER(rt._abi.rt_camera)
    syms = subprocess.run(["nm", "-D", "--defined-only", rt._abi.lib_path()], check=True, capture_output=True, text=True).stdout
    assert any(line.split()[-1] == "rt_gpu_render_view" for line in syms.splitlines())


def test_look_at(rt):
    c = rt.look_at((0, 0, 7), (0, 0, 0))
    assert isinstance(c, rt.rt_camera)
    assert list(c.eye) == [0.0, 0.0, 7.0]
    assert (list(c.right), list(c.up), list(c.back)) == ([1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0])
    assert c.dir_z == np.float32(-0.5) and c.ray_distance == 1000.0
    # an orthonormal, right-handed basis whose -back looks at the target; float64 rounded to float32
    eye, tgt = np.array([3.0, 2.0, -5.0]), np.array([0.5, -1.0, 0.25])
    c = rt.look_at(eye, tgt, up=(0.1, 1.0, 0.0), dir_z=-0.8, ray_distance=42.0)
    B = np.array([list(c.right), list(c.up), list(c.back)], np.float64)
    assert np.allclose(B @ B.T, np.eye(3), atol=1e-6) and np.linalg.det(B) > 0
    want_back = (eye - tgt) / np.linalg.norm(eye - tgt)
    assert np.array_equal(np.float32(want_back), np.array(list(c.back), np.float32))
    assert c.dir_z == np.float32(-0.8) and c.ray_distance == 42.0
    # degenerate inputs
    for args in (((1, 2, 3), (1, 2, 3)), ((0, 5, 0), (0, 0, 0)), ((0, 0, 7), (0, 0, 0), (0, 0, 3)),
                 ((0, 0, 7), (0, 0, 0), (0, 0, 0)), ((0, 0, float("nan")), (0, 0, 0))):
        with pytest.raises(ValueError):
            rt.look_at(*args)
    # raw values go through as given
    c = rt.camera((1, 2, 3), (1.5, 0, 0), (0, 2, 0), (0, 0, -1), dir_z=-0.25, ray_distance=7.0)
    assert (list(c.eye), list(c.right), list(c.up), list(c.back)) == ([1, 2, 3], [1.5, 0, 0], [0, 2, 0], [0, 0, -1])
    assert (c.dir_z, c.ray_distance) == (-0.25, 7.0)


# ---------------------------------------------------------------------------------------------------
# 1. without a camera nothing changes
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["c3_unitychan", "deterministic_mix"])
def test_no_camera_is_render_tile(rt, gpu, data_dir, scene_name):
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    d = sc.desc.contents
    same_view = rt.camera(list(d.eye), (1, 0, 0), (0, 1, 0), (0, 0, 1), d.dir_z, d.ray_distance)
    signed_zeros = rt.camera(list(d.eye), (1, -0.0, -0.0), (-0.0, 1, 0), (-0.0, -0.0, 1), d.dir_z, d.ray_distance)
    W, H = 160, 120
    for mode in (PATH, PREVIEW, WHITTED, PRIMARY):
        for aa in (0, 1):
            for tr in (EXACT, CULLED):
                p = rt.make_params(W, H, mode=mode, max_bounce=6, antialias=aa, pass_begin=1, pass_count=2, seed=5, traverse=tr)
                want = render(rt, gpu, p, False)
                for cam in (None, same_view, signed_zeros):
                    got = render(rt, gpu, p, cam)
                    assert not (diff := same_frame(got, want)), (scene_name, mode, aa, tr, list(cam.right) if cam else None, diff)
                assert want["counters"]["camera_rays"] > 0


# ---------------------------------------------------------------------------------------------------
# 2. against the restatement
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["c1_torusknot", "c2_monkey", "c2_monkey_null", "deterministic_mix", "c3_unitychan"])
def test_against_restatement(rt, gpu, view_restatement, data_dir, scene_name):
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    W, H = 160, 120
    pixels = np.arange(W * H, dtype=np.int32)
    sky_share = {}
    for cname, cam in cameras(rt, sc).items():
        for mode, aa, bounce in ((PATH, 1, 6), (PREVIEW, 1, 6), (WHITTED, 0, 1), (PRIMARY, 0, 1)):
            p = rt.make_params(W, H, mode=mode, max_bounce=bounce, antialias=aa, pass_begin=2, pass_count=1, seed=9,
                               traverse=EXACT)
            want = view_restatement.render(sc.desc, p, cam)
            wc = want["counters"]
            for tr in (EXACT, CULLED):
                p.traverse = tr
                got = render(rt, gpu, p, cam)
                c = got["counters"]
                where = (scene_name, cname, mode, tr)
                if mode in (PATH, WHITTED):
                    assert same_bits(got["accum"], want["accum"]), where
                elif mode == PREVIEW:
                    assert same_bits(got["preview"][..., :3], want["preview"][..., :3]), where
                else:
                    np.testing.assert_array_equal(got["ids"], want["ids"], err_msg=str(where))
                    assert same_bits(got["dist"], want["dist"]), where
                assert c["camera_rays"] == wc["camera_rays"] == W * H * (4 if aa else 1), where
                assert c["rays"] == wc["rays"] and c["shadow_rays"] == wc["shadow_rays"], where
                if tr == EXACT:
                    for k in ("node_tests", "tri_tests", "mesh_walks"):
                        assert c[k] == wc[k], (where, k)
            if mode == PRIMARY:
                # the same rays as nearest-hit queries
                rays, draws = view_restatement.view_rays(p, cam, pixels, -1)
                assert not draws.any()
                q = gpu.query_rays(to_dev(rays), traverse=EXACT)
                np.testing.assert_array_equal(q["shape"].cpu().numpy(), got["ids"][..., 0].reshape(-1))
                np.testing.assert_array_equal(q["tri"].cpu().numpy(), got["ids"][..., 1].reshape(-1))
                hit = q["hit"].cpu().numpy()
                assert same_bits(np.where(q["shape"].cpu().numpy() >= 0, hit[:, 6], 0.0), got["dist"].reshape(-1))
                sky_share[cname] = float((q["shape"].cpu().numpy() < 0).mean())
    # the cameras do what their names say
    assert sky_share["steep_up"] > 0.5
    assert sky_share["orbit"] < 0.95 and sky_share["zero_components"] < 0.95 and sky_share["non_orthonormal"] < 0.95


# ---------------------------------------------------------------------------------------------------
# 3. fuzzy reflection: the render's statistical bar, and radiance_rays of the same rays
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_default_scene(rt, gpu, view_restatement, data_dir):
    """Fuzzy reflection calls sinf / cosf / acosf, whose CUDA and glibc results differ in the last ulp: against the
    restatement the render's bar (>= 99.8 % of pixels within 1e-4, the mean within 0.1 %); against GPU radiance_rays
    of the camera's own rays (stream = pixel, sample = 4 pass + sub, first draw 2) bit for bit."""
    sc = scene_of(rt, "default_scene", data_dir)
    gpu.upload_scene(sc)
    W, H = 160, 120
    pixels = np.arange(W * H, dtype=np.int32)
    cams = cameras(rt, sc)
    for cname in ("orbit", "non_orthonormal", "steep_down"):
        cam = cams[cname]
        p = rt.make_params(W, H, mode=PATH, max_bounce=6, antialias=1, pass_begin=3, pass_count=1, seed=4)
        got = render(rt, gpu, p, cam)["accum"].reshape(-1, 4)
        want = view_restatement.render(sc.desc, p, cam)["accum"].reshape(-1, 4)
        bad = (np.abs(got[:, :3] - want[:, :3]) > 1e-4).any(1) | (np.isnan(got[:, :3]) != np.isnan(want[:, :3])).any(1)
        assert bad.mean() <= 2e-3, (cname, bad.mean())
        ok = np.isfinite(got[:, :3]).all(1) & np.isfinite(want[:, :3]).all(1)
        assert abs(got[ok, :3].mean() - want[ok, :3].mean()) <= 1e-3 * want[ok, :3].mean(), cname
        col = np.zeros((W * H, 3), np.float32)
        for i in range(4):
            rays, draws = view_restatement.view_rays(p, cam, pixels, i)
            assert (draws == 2).all()
            col = col + gpu.radiance_rays(to_dev(rays), mode=PATH, max_bounce=6, seed=4, sample=4 * 3 + i,
                                          rng_stream=to_dev(pixels), first_draw=2).cpu().numpy()[:, :3]
        assert same_bits(np.float32(0.0) + col / np.float32(4.0), got[:, :3]), cname


# ---------------------------------------------------------------------------------------------------
# 4.-6. passes, tiles, frame slots
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_passes_and_retry_passes(rt, gpu, data_dir):
    """pass_begin > 0 and pass_count > 1 in one call, with pools so small that retry passes run, equal the same passes
    one call each on default pools."""
    sc = scene_of(rt, "c3_unitychan", data_dir)
    cam = cameras(rt, sc)["orbit"]
    W, H = 160, 120
    small = rt.GpuContext(0)
    small.set_tuning(pool_kpaths=8)
    small.upload_scene(sc)
    gpu.upload_scene(sc)
    for mode in (PATH, PREVIEW):
        p = rt.make_params(W, H, mode=mode, max_bounce=6, antialias=1, pass_begin=3, pass_count=5, seed=2)
        whole = render(rt, small, p, cam)
        gpu.reset_accum(W, H)
        gpu.synchronize()
        gpu.reset_counters()
        gpu.synchronize()
        for k in range(5):
            gpu.render_tile(rt.make_params(W, H, mode=mode, max_bounce=6, antialias=1, pass_begin=3 + k, pass_count=1, seed=2), cam)
        gpu.synchronize()
        parts = read_all(rt, gpu, W, H, preview=mode == PREVIEW)
        assert not (diff := same_frame(whole, parts)), (mode, diff)
        assert whole["counters"]["camera_rays"] == 5 * 4 * W * H
    small.close()


@pytest.mark.gpu
def test_tiles(rt, gpu, data_dir):
    import torch
    sc = scene_of(rt, "deterministic_mix", data_dir)
    gpu.upload_scene(sc)
    cam = cameras(rt, sc)["non_orthonormal"]
    W, H = 160, 120
    kw = dict(mode=PATH, max_bounce=5, antialias=1, pass_count=2, seed=6)
    full = render(rt, gpu, rt.make_params(W, H, **kw), cam)
    for n in (2, 4, 8):
        dense = []
        for r in range(n):
            p = rt.make_params(W, H, tile_size=16, tile_count=n, tile_rank=r, **kw)
            gpu.reset_accum(W, H)
            gpu.render_tile(p, cam)
            buf = torch.empty((rt.owned_pixels(W, H, 16, n, r), 4), dtype=torch.float32, device="cuda:0")
            gpu.pack_owned(p, buf.data_ptr(), buf.numel() * 4)
            gpu.synchronize()
            dense.append((p, buf))
        gpu.reset_accum(W, H)
        for r, (p, buf) in enumerate(dense):
            gpu.unpack_owned(p, r, buf.data_ptr(), buf.numel() * 4)
        gpu.synchronize()
        assert np.array_equal(bits(gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(full["accum"])), n


@pytest.mark.gpu
def test_frame_slots(rt, data_dir):
    """Four slots, each its own camera, enqueued back to back with no synchronisation, equal each camera rendered alone
    on a fresh context; a render_tile afterwards equals a fresh context's (no camera state is kept)."""
    sc = scene_of(rt, "c3_unitychan", data_dir)
    cams = list(cameras(rt, sc).values())[:4]
    W, H = 160, 120
    p = rt.make_params(W, H, mode=PATH, max_bounce=6, antialias=1, pass_count=2, seed=8)
    reads = dict(accum=rt.RT_READ_ACCUM_RGBN_F32, display=rt.RT_READ_DISPLAY_ARGB8)
    want = []
    for cam in cams:
        ctx = rt.GpuContext(0)
        ctx.upload_scene(sc)
        want.append(render(rt, ctx, p, cam, reads))
        ctx.close()
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)
    for s in range(4):
        ctx.set_frame_slot(s)
        ctx.reset_accum(W, H)
    for s, cam in enumerate(cams):
        ctx.set_frame_slot(s)
        ctx.render_tile(p, cam)
    for s in range(4):
        ctx.set_frame_slot(s)
        ctx.synchronize()
        got = {k: ctx.readback(w, W, H).copy() for k, w in reads.items()}
        for k in reads:
            assert np.array_equal(got[k].view(np.uint8), want[s][k].view(np.uint8)), (s, k)
    ctx.set_frame_slot(0)
    after = render(rt, ctx, p, False, reads)
    fresh = rt.GpuContext(0)
    fresh.upload_scene(sc)
    assert not (diff := same_frame(after, render(rt, fresh, p, False, reads))), diff
    fresh.close()
    ctx.close()


# ---------------------------------------------------------------------------------------------------
# 7. bad input changes nothing
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_input(rt, data_dir):
    abi = rt._abi
    lib = rt.load_library()
    sc = scene_of(rt, "deterministic_mix", data_dir)
    W, H = 96, 64
    p = rt.make_params(W, H, mode=PATH, max_bounce=4, antialias=1, pass_count=1, seed=1)
    good = rt.look_at((1.0, 1.0, 6.0), (0.0, 0.0, 0.0))
    ctx = rt.GpuContext(0)
    assert lib.rt_gpu_render_view(ctx.handle, C.byref(p), C.byref(good)) == abi.RT_ERR_NO_SCENE
    assert lib.rt_gpu_last_error(ctx.handle)
    with pytest.raises(rt.RtError):
        ctx.render_tile(p, good)
    ctx.upload_scene(sc)
    ctx.reset_accum(W, H)
    ctx.render_tile(p, good)
    ctx.synchronize()
    before = read_all(rt, ctx, W, H)
    assert before["counters"]["camera_rays"] > 0

    def unchanged():
        ctx.synchronize()
        assert not (diff := same_frame(read_all(rt, ctx, W, H), before)), diff

    def copy(cam):
        c = rt.rt_camera()
        C.memmove(C.byref(c), C.byref(cam), C.sizeof(c))
        return c

    bad = []
    for f in ("eye", "right", "up", "back"):
        for i in range(3):
            for v in (float("nan"), float("inf"), float("-inf")):
                c = copy(good)
                getattr(c, f)[i] = v
                bad.append(c)
    for f in ("dir_z", "ray_distance"):
        for v in (float("nan"), float("inf"), float("-inf")):
            c = copy(good)
            setattr(c, f, v)
            bad.append(c)
    bad.append(rt.camera((0, 0, 7), (0, 0, 0), (0, 0, 0), (0, 0, 0)))                 # zero basis
    bad.append(rt.camera((0, 0, 7), (1, 0, 0), (0, 1, 0), (0, 0, 0)))                 # a zero vector
    bad.append(rt.camera((0, 0, 7), (1, 2, 3), (2, 4, 6), (0, 0, 1)))                 # right parallel to up
    bad.append(rt.camera((0, 0, 7), (1, 0, 0), (0, 1, 0), (1, 1, 0)))                 # back in the plane of the others
    for c in bad:
        assert lib.rt_gpu_render_view(ctx.handle, C.byref(p), C.byref(c)) == abi.RT_ERR_INVALID
        assert lib.rt_gpu_last_error(ctx.handle)
        with pytest.raises(rt.RtError):
            ctx.render_tile(p, c)
        unchanged()
    # the usual bad params, with a good camera
    for kw in (dict(mode=7), dict(traverse=2), dict(max_bounce=-1), dict(max_bounce=33), dict(pass_count=-1),
               dict(pass_begin=-1), dict(start=-1), dict(end=W * H), dict(tile_count=2, tile_size=0)):
        q = rt.make_params(W, H, mode=PATH, max_bounce=4, antialias=1, pass_count=1, seed=1)
        for k, v in kw.items():
            setattr(q, k, v)
        assert lib.rt_gpu_render_view(ctx.handle, C.byref(q), C.byref(good)) == abi.RT_ERR_INVALID, kw
        with pytest.raises(rt.RtError):
            ctx.render_tile(q, good)
        unchanged()
    assert lib.rt_gpu_render_view(ctx.handle, None, C.byref(good)) == abi.RT_ERR_INVALID
    with pytest.raises(TypeError):
        ctx.render_tile(p, (0, 0, 7))
    unchanged()
    # still usable: the same call renders the same frame on top
    ctx.render_tile(p, good)
    ctx.synchronize()
    acc = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert np.array_equal(acc[..., 3], 2 * before["accum"][..., 3])
    ctx.close()
