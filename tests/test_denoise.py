"""The guided denoiser: the RT_MODE_GUIDES render mode (first-hit ids, distance and normal per pixel) and
rt_gpu_denoise / GpuContext.denoise, the edge-avoiding a-trous filter of include/rt_gpu.h.

GUIDES is held to RT_MODE_PRIMARY (ids and distance, counters) and to the nearest-hit queries of rt_gpu_query_rays on
the render's own camera rays (normals), bit for bit.  The filter is held bit for bit to `restate`, a numpy float32
restatement of the header's formula (one rounding per operation, in the header's order), which the CPU tests check on
hand-built frames."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT, same_bits
from test_adaptive_sampling import dev, fresh, scene_of, turned_camera

PATH, PREVIEW, WHITTED, PRIMARY, GUIDES = 0, 1, 2, 3, 4
EXACT, CULLED = 0, 1
F32 = np.float32
H5 = np.array([0.0625, 0.25, 0.375, 0.25, 0.0625], F32)
DEFAULTS = dict(levels=5, normal_log2=7, sigma_lum=4.0, sigma_depth=0.1, lum_floor=0.02)
STABLE_COUNTERS = ("rays", "camera_rays", "shadow_rays", "mesh_hits", "mesh_walks")


# ---------------------------------------------------------------------------------------------------
# the restatement
# ---------------------------------------------------------------------------------------------------
def lum(v):
    """Y(v) = (0.2126f*r + 0.7152f*g) + 0.0722f*b over the last axis, float32"""
    return (F32(0.2126) * v[..., 0] + F32(0.7152) * v[..., 1]) + F32(0.0722) * v[..., 2]


def restate(acc, shape, z, nrm, preview=None, moments=None, levels=5, normal_log2=7, sigma_lum=4.0, sigma_depth=0.1,
            lum_floor=0.02):
    """rgba (H, W, 4) of rt_gpu_denoise: acc = accuBuffer (H, W, 4), shape / z = the primary shape ids and distances (H, W),
    nrm = the guide normals (H, W, 3+); preview (H, W, 3+) with use_albedo, moments (H, W, 4) with use_variance."""
    acc = np.asarray(acc, F32)
    Hh, Ww = acc.shape[:2]
    z = np.asarray(z, F32)
    nrm = np.asarray(nrm, F32)[..., :3]
    shape = np.asarray(shape, np.int64)
    with np.errstate(all="ignore"):
        n = acc[..., 3].astype(np.int64)
        fn = n.astype(F32)
        finite = np.isfinite(acc[..., :3]).all(-1)
        valid = (n > 0) & finite
        c = acc[..., :3] / fn[..., None]
        if preview is not None:
            a = np.asarray(preview, F32)[..., :3]
            d = np.where(a > F32(1e-3), a, F32(1e-3)).astype(F32)
        else:
            d = np.ones((Hh, Ww, 3), F32)
        x = np.where(valid[..., None], c / d, F32(0)).astype(F32)
        v = np.zeros((Hh, Ww), F32)
        if moments is not None:
            m = np.asarray(moments, F32)
            vv = (lum(m[..., :3]) / (n - 1).astype(F32)) / fn
            if preview is not None:
                yd = lum(d)
                vv = vv / (yd * yd)
            v = np.where(valid & (n >= 2) & (m[..., 3] == fn), vv, F32(0)).astype(F32)
        sh = np.where(valid, shape, -2)
        hit = sh >= 0
        yy, xx = np.mgrid[0:Hh, 0:Ww]
        for k in range(levels):
            s = 1 << k
            yp = lum(x)
            lum_scale = F32(sigma_lum) * np.sqrt(v) + F32(lum_floor)
            depth_scale = (F32(sigma_depth) * F32(s)) * z
            W = np.zeros((Hh, Ww), F32)
            V = np.zeros((Hh, Ww), F32)
            X = np.zeros((Hh, Ww, 3), F32)
            for j in range(-2, 3):
                for i in range(-2, 3):
                    qy, qx = yy + s * j, xx + s * i
                    inside = (qy >= 0) & (qy < Hh) & (qx >= 0) & (qx < Ww)
                    qy, qx = np.clip(qy, 0, Hh - 1), np.clip(qx, 0, Ww - 1)
                    xq, vq = x[qy, qx], v[qy, qx]
                    if i == 0 and j == 0:
                        w = np.full((Hh, Ww), F32(0.140625))
                        take = valid
                    else:
                        take = valid & inside & (sh[qy, qx] == sh)
                        h = H5[i + 2] * H5[j + 2]
                        nq, zq = nrm[qy, qx], z[qy, qx]
                        wn = (nrm[..., 0] * nq[..., 0] + nrm[..., 1] * nq[..., 1]) + nrm[..., 2] * nq[..., 2]
                        wn = np.where(wn > F32(0), wn, F32(0)).astype(F32)
                        for _ in range(normal_log2):
                            wn = wn * wn
                        wz = F32(1) / (F32(1) + np.abs(z - zq) / depth_scale)
                        w = np.where(hit, (h * wn) * wz, h).astype(F32)
                        t = np.abs(yp - lum(xq)) / lum_scale
                        w = w * (F32(1) / (F32(1) + t * t))
                        take = take & np.isfinite(w)
                    W = np.where(take, W + w, W)
                    X = np.where(take[..., None], X + w[..., None] * xq, X)
                    V = np.where(take, V + (w * w) * vq, V)
            x = np.where(valid[..., None], X / W[..., None], x).astype(F32)
            v = np.where(valid, V / (W * W), v).astype(F32)
        out = np.zeros((Hh, Ww, 4), F32)
        rgb = np.where(finite[..., None], x * d, c)
        out[..., :3] = np.where((n > 0)[..., None], rgb, F32(0))
        out[..., 3] = np.where(n > 0, fn, F32(0))
    return out


# ---------------------------------------------------------------------------------------------------
# no GPU: layout, bindings and the restatement on hand-built frames
# ---------------------------------------------------------------------------------------------------
def test_denoise_params_layout_matches_c(rt):
    fields = ("levels", "use_albedo", "use_variance", "normal_log2", "sigma_lum", "sigma_depth", "lum_floor")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rt_gpu.h\"\nint main(void) {\n"
    src += '  printf("size %zu\\n", sizeof(rt_denoise_params));\n'
    src += '  printf("guides %d\\n", (int)RT_MODE_GUIDES);\n'
    src += '  printf("guide_read %d\\n", (int)RT_READ_GUIDE_NORMAL_F32);\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_denoise_params, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "q.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "q")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    dp = rt._abi.rt_denoise_params
    assert C.sizeof(dp) == out["size"] == 28
    for f in fields:
        assert getattr(dp, f).offset == out[f], f
    assert rt.RT_MODE_GUIDES == out["guides"] == 4
    assert rt.RT_READ_GUIDE_NORMAL_F32 == out["guide_read"] == 7


def test_denoise_calls_are_bound(rt):
    lib = rt.load_library()
    for name in ("rt_gpu_denoise", "rt_gpu_frame_size"):
        assert name in rt._abi.GPU_PROTOTYPES
        assert getattr(lib, name).restype is C.c_int
    assert lib.rt_gpu_denoise.argtypes[1] is C.POINTER(rt._abi.rt_denoise_params)


def _flat_guides(Hh, Ww, shape=0):
    return np.full((Hh, Ww), shape, np.int64), np.full((Hh, Ww), F32(3.0)), np.tile(np.array([0, 0, 1], F32), (Hh, Ww, 1))


def test_restatement_keeps_a_constant_frame():
    Hh, Ww = 24, 40
    acc = np.zeros((Hh, Ww, 4), F32)
    acc[..., :3] = np.array([0.3, 0.55, 0.2], F32) * F32(6)
    acc[..., 3] = 6
    mom = np.zeros((Hh, Ww, 4), F32)
    mom[..., :3], mom[..., 3] = F32(0.01), 6
    alb = np.tile(np.array([0.5, 0.7, 0.9], F32), (Hh, Ww, 1))
    shape, z, nrm = _flat_guides(Hh, Ww)
    want = acc[..., :3] / F32(6)
    for levels in (1, 3, 6):
        for preview, moments in ((None, None), (alb, None), (None, mom), (alb, mom)):
            out = restate(acc, shape, z, nrm, preview, moments, levels=levels)
            # a weighted mean of equal values: each level can move it by an ulp or two
            assert np.allclose(out[..., :3], want, rtol=8 * np.finfo(F32).eps, atol=0), (levels, preview is None, moments is None)
            assert (out[..., 3] == 6).all()


def test_restatement_leaks_nothing_across_a_shape_edge():
    Hh, Ww = 32, 32
    rng = np.random.default_rng(3)
    acc = np.zeros((Hh, Ww, 4), F32)
    acc[..., 3] = 4
    acc[:, :16, :3] = rng.random((Hh, 16, 3), dtype=F32) * F32(4)     # noisy left half
    acc[:, 16:, :3] = F32(40)                                          # bright constant right half
    shape = np.zeros((Hh, Ww), np.int64)
    shape[:, 16:] = 1
    _, z, nrm = _flat_guides(Hh, Ww)
    out = restate(acc, shape, z, nrm, levels=5, lum_floor=1e6)         # luminance weight ~1: only the ids separate
    assert (out[:, 16:, :3] == F32(10)).all()
    assert (out[:, :16, :3] < F32(1.0001)).all()
    # with one id everywhere the bright half does leak (the check above is not vacuous)
    out1 = restate(acc, np.zeros((Hh, Ww), np.int64), z, nrm, levels=5, lum_floor=1e6)
    assert (out1[:, 12:16, :3] > F32(1.5)).all()


def test_restatement_output_rules_for_invalid_pixels():
    Hh, Ww = 16, 20
    rng = np.random.default_rng(5)
    acc = np.zeros((Hh, Ww, 4), F32)
    acc[..., :3] = rng.random((Hh, Ww, 3), dtype=F32) * F32(3)
    acc[..., 3] = 3
    acc[2, 3, 3] = 0                           # no passes
    acc[2, 3, :3] = 7
    acc[5, 6, 1] = np.nan                      # a NaN sum
    acc[7, 8, 2] = np.inf                      # an infinite sum
    shape, z, nrm = _flat_guides(Hh, Ww)
    shape[10:, :] = -1                         # misses: the normal and depth weights are left out
    alb = rng.random((Hh, Ww, 3), dtype=F32)
    for preview in (None, alb):
        out = restate(acc, shape, z, nrm, preview, levels=4)
        assert (out[2, 3] == 0).all()
        with np.errstate(all="ignore"):
            assert same_bits(out[5, 6, :3], acc[5, 6, :3] / F32(3)) and same_bits(out[7, 8, :3], acc[7, 8, :3] / F32(3))
        assert out[5, 6, 3] == 3 and out[7, 8, 3] == 3
        good = np.ones((Hh, Ww), bool)
        good[2, 3] = good[5, 6] = good[7, 8] = False
        assert np.isfinite(out[good]).all()
        # an invalid pixel is no tap of its neighbours: the frame without them filters its other pixels the same way
        acc2 = acc.copy()
        acc2[2, 3, :3] = 1000
        acc2[5, 6, :3] = np.nan
        acc2[7, 8, :3] = (-np.inf, 5, 5)
        out2 = restate(acc2, shape, z, nrm, preview, levels=4)
        assert same_bits(out2[good], out[good])


# ---------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------
def params(rt, w, h, **kw):
    base = dict(mode=PATH, max_bounce=6, antialias=1, seed=3, traverse=CULLED)
    base.update(kw)
    return rt.make_params(w, h, **base)


def guides(rt, ctx, w, h):
    ids = ctx.readback(rt.RT_READ_PRIMARY_IDS_I32X2, w, h).copy()
    dist = ctx.readback(rt.RT_READ_PRIMARY_DIST_F32, w, h).copy()
    nrm = ctx.readback(rt.RT_READ_GUIDE_NORMAL_F32, w, h).copy()
    return ids, dist, nrm


def frame_state(rt, ctx, w, h, preview=True, moments=True):
    s = dict(accum=ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h).copy(),
             display=ctx.readback(rt.RT_READ_DISPLAY_ARGB8, w, h).copy())
    if preview:
        s["preview"] = ctx.readback(rt.RT_READ_PREVIEW_RGBA_F32, w, h).copy()
    if moments:
        s["moments"] = ctx.readback(rt.RT_READ_MOMENTS_F32, w, h).copy()
    return s


def same_state(a, b):
    return a.keys() == b.keys() and all(np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)) for k in a)


def kat_pixels(rt, ctx, rgb):
    """MakePixelColor(LinearToGamma(rgb)) of the device (rt_gpu_kat kind 7), uint32"""
    rgb = np.ascontiguousarray(rgb, F32).reshape(-1, 3)
    flags = np.zeros(len(rgb), np.int32)
    out7 = np.zeros((len(rgb), 7), F32)
    assert rt.load_library().rt_gpu_kat(ctx.handle, 7, None, rgb.ctypes.data, 3, len(rgb), flags.ctypes.data, out7.ctypes.data) == 0
    return flags.view(np.uint32)


def prepared_frame(rt, ctx, w, h, cam=None, seed=3, max_bounce=6, holes=True):
    """A PATH frame with passes that differ per pixel, moments that cover only some of them, a PREVIEW pass and a GUIDES
    render; with holes, some pixels get n = 0 and some a NaN or infinite sum (written back through unpack_owned)."""
    import torch
    fresh(ctx, w, h)
    rng = np.random.default_rng(seed)
    p = params(rt, w, h, seed=seed, max_bounce=max_bounce)
    ctx.track_moments(True)
    p.pass_begin, p.pass_count = 0, 3
    ctx.render_tile(p, cam)
    p.pass_begin, p.pass_count = 3, 3
    ctx.render_tile(p, cam, mask=dev((rng.random((h, w)) < 0.6).astype(np.uint8)))
    ctx.track_moments(False)                                  # this pass is not in the moments
    p.pass_begin, p.pass_count = 6, 1
    ctx.render_tile(p, cam, mask=dev((rng.random((h, w)) < 0.3).astype(np.uint8)))
    if holes:
        acc = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h).copy()
        acc[rng.random((h, w)) < 0.03] = 0
        acc[rng.random((h, w)) < 0.02, 1] = np.nan
        acc[rng.random((h, w)) < 0.01, 0] = np.inf
        buf = dev(acc)
        torch.cuda.synchronize()
        ctx.unpack_owned(params(rt, w, h), 0, buf.data_ptr(), buf.numel() * 4)
    ctx.render_tile(params(rt, w, h, mode=PREVIEW, pass_begin=0, pass_count=1, seed=seed), cam)
    ctx.render_tile(params(rt, w, h, mode=GUIDES), cam)
    ctx.synchronize()


def inputs(rt, ctx, w, h):
    ids, dist, nrm = guides(rt, ctx, w, h)
    s = frame_state(rt, ctx, w, h)
    return dict(acc=s["accum"], shape=ids[..., 0], z=dist, nrm=nrm, preview=s["preview"], moments=s["moments"])


def denoised(ctx, **kw):
    import torch
    out, pix = ctx.denoise(argb=True, **kw)
    torch.cuda.synchronize()
    return out.cpu().numpy(), pix.cpu().numpy().view(np.uint32)


def check_denoise(rt, ctx, d, w, h, albedo, variance, **kw):
    prm = dict(DEFAULTS, **kw)
    got, pix = denoised(ctx, use_albedo=albedo, use_variance=variance, **prm)
    want = restate(d["acc"], d["shape"], d["z"], d["nrm"], d["preview"] if albedo else None, d["moments"] if variance else None, **prm)
    where = (albedo, variance, prm)
    assert same_bits(got, want), where
    n = d["acc"][..., 3]
    assert (pix[n <= 0] == 0).all(), where
    assert np.array_equal(pix[n > 0], kat_pixels(rt, ctx, want[n > 0][:, :3])), where
    return got


# ---------------------------------------------------------------------------------------------------
# GUIDES
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["default_scene", "c3_unitychan"])
def test_guides_are_primary_plus_normals(rt, gpu, data_dir, scene_name):
    """ids and distance equal PRIMARY's, with and without a camera, for sub-ranges, tiles and masks; the counters equal
    PRIMARY's; accum, display, moments and preview keep their bytes; the normals of pixels outside the task stay zero"""
    w, h = 192, 108
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    cam = turned_camera(rt, sc)
    rng = np.random.default_rng(7)
    some = dev((rng.random((h, w)) < 0.5).astype(np.uint8))
    tasks = dict(full={}, sub_range=dict(start=w * 17 + 5, end=w * 93 + 130), tiles=dict(tile_size=16, tile_count=3, tile_rank=1))
    for tr in (EXACT, CULLED):
        for tname, tkw in tasks.items():
            for c in (None, cam):
                for mask in (None, some):
                    runs = {}
                    for mode in (PRIMARY, GUIDES):
                        # a frame with accumulated passes, moments and a preview colour first
                        gpu.set_frame_slot(0)
                        fresh(gpu, w, h)
                        gpu.render_tile(params(rt, w, h, pass_count=2, traverse=tr), c)
                        gpu.track_moments(True)
                        gpu.render_tile(params(rt, w, h, pass_begin=2, pass_count=2, traverse=tr), c)
                        gpu.track_moments(False)
                        gpu.render_tile(params(rt, w, h, mode=PREVIEW, traverse=tr), c)
                        gpu.synchronize()
                        before = frame_state(rt, gpu, w, h)
                        gpu.reset_counters()
                        # GUIDES ignores antialias and pass_count: give it both
                        q = params(rt, w, h, mode=mode, traverse=tr, antialias=1 if mode == GUIDES else 0,
                                   pass_begin=3, pass_count=5 if mode == GUIDES else 1, **tkw)
                        gpu.render_tile(q, c, mask=mask)
                        gpu.synchronize()
                        assert same_state(frame_state(rt, gpu, w, h), before), (mode, tr, tname)
                        runs[mode] = (gpu.readback(rt.RT_READ_PRIMARY_IDS_I32X2, w, h).copy(),
                                      gpu.readback(rt.RT_READ_PRIMARY_DIST_F32, w, h).copy(), gpu.counters())
                    where = (tr, tname, c is not None, mask is not None)
                    assert np.array_equal(runs[GUIDES][0], runs[PRIMARY][0]), where
                    assert same_bits(runs[GUIDES][1], runs[PRIMARY][1]), where
                    for k in (runs[PRIMARY][2] if tr == EXACT else STABLE_COUNTERS):
                        assert runs[GUIDES][2][k] == runs[PRIMARY][2][k], (where, k)
                    assert runs[GUIDES][2]["camera_rays"] > 0
                    nrm = gpu.readback(rt.RT_READ_GUIDE_NORMAL_F32, w, h)
                    assert (nrm[..., 3] == 0).all()
                    if tname == "full" and mask is None:
                        ids = runs[GUIDES][0][..., 0]
                        assert (nrm[ids < 0] == 0).all() and (ids < 0).any(), where
                        assert (nrm[ids >= 0] != 0).any(-1).all(), where


@pytest.fixture(scope="module")
def restatement(tmp_path_factory):
    """the camera rays of render_tile, restated (tests/test_radiance_queries.py)"""
    from test_radiance_queries import RADIANCE_SRC, Restatement
    d = tmp_path_factory.mktemp("denoise_rays")
    src, lib = d / "radiance.c", d / "libradiance.so"
    src.write_text(RADIANCE_SRC)
    subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                    "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"),
                    "-o", str(lib), str(src), "-lm", "-lpthread"], check=True)
    L = C.CDLL(str(lib))
    L.camera_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return Restatement(L)


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["default_scene", "c2_monkey", "c3_unitychan", "deterministic_mix"])
def test_guide_normals_are_the_query_hits(rt, gpu, restatement, data_dir, scene_name):
    """the normal of each pixel is the HitNormal rt_gpu_query_rays reports for the pixel's un-jittered camera ray"""
    import torch
    w, h = 256, 144
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    for tr in (EXACT, CULLED):
        fresh(gpu, w, h)
        p = params(rt, w, h, mode=GUIDES, traverse=tr)
        gpu.render_tile(p)
        gpu.synchronize()
        ids, dist, nrm = guides(rt, gpu, w, h)
        rays, _ = restatement.camera_rays(sc.desc, p, np.arange(w * h, dtype=np.int32), -1)
        r = gpu.query_rays(torch.from_numpy(rays).to("cuda:0"), traverse=tr)
        torch.cuda.synchronize()
        shape, hit = r["shape"].cpu().numpy(), r["hit"].cpu().numpy()
        assert np.array_equal(shape, ids[..., 0].reshape(-1)), (scene_name, tr)
        assert same_bits(hit[:, 3:6], nrm[..., :3].reshape(-1, 3)), (scene_name, tr)
        assert same_bits(np.where(shape >= 0, hit[:, 6], 0), dist.reshape(-1)), (scene_name, tr)
        assert (nrm[..., 3] == 0).all() and (shape >= 0).any()


# ---------------------------------------------------------------------------------------------------
# the filter
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["default_scene", "c2_monkey", "c3_unitychan"])
def test_denoise_equals_the_restatement(rt, gpu, data_dir, scene_name):
    w, h = 192, 108
    sc = scene_of(rt, scene_name, data_dir)
    gpu.upload_scene(sc)
    gpu.set_frame_slot(0)
    prepared_frame(rt, gpu, w, h)
    d = inputs(rt, gpu, w, h)
    n = d["acc"][..., 3]
    assert (n == 0).any() and np.isnan(d["acc"][..., 1]).any() and len(np.unique(n)) >= 4
    assert len(np.unique(d["shape"])) >= 2
    assert ((d["moments"][..., 3] == n) & (n >= 2)).any() and (d["moments"][..., 3] != n).any()
    for levels in range(1, 7):
        for albedo in (False, True):
            for variance in (False, True):
                check_denoise(rt, gpu, d, w, h, albedo, variance, levels=levels)
    # other weights
    check_denoise(rt, gpu, d, w, h, True, True, levels=3, normal_log2=0, sigma_lum=0.0, sigma_depth=0.02, lum_floor=0.5)
    check_denoise(rt, gpu, d, w, h, False, True, levels=4, normal_log2=8, sigma_lum=1.5, sigma_depth=3.0, lum_floor=1e-4)


@pytest.mark.gpu
def test_denoise_moved_camera_and_path_frame_without_holes(rt, gpu, data_dir):
    w, h = 256, 144
    sc = scene_of(rt, "default_scene", data_dir)
    gpu.upload_scene(sc)
    cam = turned_camera(rt, sc)
    gpu.set_frame_slot(0)
    prepared_frame(rt, gpu, w, h, cam=cam, seed=11, holes=False)
    d = inputs(rt, gpu, w, h)
    for levels, albedo, variance in ((5, True, True), (2, False, True), (6, True, False)):
        check_denoise(rt, gpu, d, w, h, albedo, variance, levels=levels)
    # use_variance=None: the slot tracks moments
    got = gpu.denoise(use_albedo=True).cpu().numpy()
    assert same_bits(got, restate(d["acc"], d["shape"], d["z"], d["nrm"], d["preview"], d["moments"], **DEFAULTS))
    # a slot that never tracked moments filters without variance
    gpu.set_frame_slot(2)
    fresh(gpu, w, h)
    gpu.render_tile(params(rt, w, h, pass_count=3), cam)
    gpu.render_tile(params(rt, w, h, mode=GUIDES), cam)
    gpu.synchronize()
    ids, dist, nrm = guides(rt, gpu, w, h)
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h).copy()
    got = gpu.denoise().cpu().numpy()
    assert same_bits(got, restate(acc, ids[..., 0], dist, nrm, **DEFAULTS))
    gpu.set_frame_slot(0)


@pytest.mark.gpu
def test_denoise_ordering_across_slots_and_streams(rt, gpu, data_dir):
    """guides rendered on slot 1 while slot 0 renders, the result consumed on a side torch stream with no host sync"""
    import torch
    w, h = 256, 144
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    kw = dict(levels=5, use_albedo=True, use_variance=True)

    def slot1_work():
        gpu.set_frame_slot(1)
        gpu.reset_accum(w, h)
        gpu.track_moments(True)
        gpu.render_tile(params(rt, w, h, pass_count=6, seed=9))
        gpu.render_tile(params(rt, w, h, mode=PREVIEW, seed=9))
        gpu.render_tile(params(rt, w, h, mode=GUIDES))

    slot1_work()
    gpu.synchronize()
    torch.cuda.synchronize()
    want = gpu.denoise(**kw).cpu().numpy()
    # again, with slot 0 busy and the output read on a side stream
    gpu.set_frame_slot(0)
    gpu.reset_accum(1920, 1080)
    gpu.render_tile(params(rt, 1920, 1080, pass_count=8, max_bounce=10))
    slot1_work()
    side = torch.cuda.Stream(device="cuda:0")
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        out = gpu.denoise(**kw)
        twice = out * 2
    side.synchronize()
    assert same_bits(twice.cpu().numpy() / F32(2), want)
    gpu.set_frame_slot(0)
    gpu.synchronize()


@pytest.mark.gpu
def test_denoise_beats_the_raw_frame(rt, gpu, data_dir):
    """8 passes, denoised, against the raw 8-pass mean: RMSE of each against the mean of 256 passes of other pass indices,
    on the framed 1080p view of tools/bench_denoise.py (the render is seeded: the figures are deterministic).  On an
    NVIDIA B200 (1000 W) with the stand-in unitychan the denoised RMSE is 0.4495 of the raw one (0.00591 against 0.01315);
    the test asks for less than 0.6.  (At 256 x 144 the same view gives only 0.91:
    there the figure's detail is a few pixels wide and the filter's footprint blurs it.)"""
    w, h = 1920, 1080
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    d = sc.desc.contents.shapes[0]
    lo, hi = np.array(list(d.bounds_min), np.float64), np.array(list(d.bounds_max), np.float64)
    center, half = (lo + hi) / 2, (hi - lo) / 2
    cam = rt.look_at(center + (0.35 * half[1] / 0.5 + max(half[0], half[2])) * np.array([0.0, 0.0, 1.0]), center)
    base = dict(max_bounce=10, seed=1)
    gpu.set_frame_slot(0)
    fresh(gpu, w, h)
    for b in range(0, 256, 32):
        gpu.render_tile(params(rt, w, h, pass_begin=100000 + b, pass_count=32, **base), cam)
    ref = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h).copy()
    ref = ref[..., :3].astype(np.float64) / ref[..., 3:4]
    fresh(gpu, w, h)
    gpu.track_moments(True)
    gpu.render_tile(params(rt, w, h, pass_count=8, **base), cam)
    gpu.render_tile(params(rt, w, h, mode=PREVIEW, **base), cam)
    gpu.render_tile(params(rt, w, h, mode=GUIDES), cam)
    gpu.synchronize()
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h).copy()
    raw = acc[..., :3].astype(np.float64) / acc[..., 3:4]
    den = gpu.denoise(use_albedo=True).cpu().numpy()[..., :3].astype(np.float64)
    e_raw = float(np.sqrt(np.mean((raw - ref) ** 2)))
    e_den = float(np.sqrt(np.mean((den - ref) ** 2)))
    print(f"RMSE raw {e_raw:.5f} denoised {e_den:.5f} ratio {e_den / e_raw:.4f}")
    assert e_den < 0.6 * e_raw


@pytest.mark.gpu
def test_refused_calls_change_nothing(rt, data_dir):
    import torch
    w, h = 192, 108
    ctx = rt.GpuContext(0)
    lib = rt.load_library()
    hd = ctx.handle
    sc = scene_of(rt, "c3_unitychan", data_dir)
    ctx.upload_scene(sc)
    out = torch.full((h, w, 4), 7.0, dtype=torch.float32, device="cuda:0")
    pix = torch.full((h, w), 7, dtype=torch.int32, device="cuda:0")
    host = np.zeros((h, w, 4), np.float32)
    prm = lambda **kw: rt._abi.rt_denoise_params(*[kw.get(k, v) for k, v in (
        ("levels", 5), ("use_albedo", 0), ("use_variance", 0), ("normal_log2", 7), ("sigma_lum", 4.0), ("sigma_depth", 0.1),
        ("lum_floor", 0.02))])
    op, pp = out.data_ptr(), pix.data_ptr()
    call = lambda p, o=None, a=None: lib.rt_gpu_denoise(hd, None if p is None else C.byref(p), op if o is None else o, pp if a is None else a, None)
    # no frame, then a frame without guides
    assert call(prm()) == rt._abi.RT_ERR_INVALID
    ctx.reset_accum(w, h)
    ctx.render_tile(params(rt, w, h, pass_count=2))
    ctx.synchronize()
    assert call(prm()) == rt._abi.RT_ERR_INVALID
    ctx.render_tile(params(rt, w, h, mode=PRIMARY))
    assert call(prm()) == rt._abi.RT_ERR_INVALID
    ctx.render_tile(params(rt, w, h, mode=GUIDES))
    ctx.synchronize()
    torch.cuda.synchronize()

    def state():
        s = frame_state(rt, ctx, w, h, preview=False, moments=False)
        s["ids"], s["dist"], s["nrm"] = guides(rt, ctx, w, h)
        s["out"], s["pix"] = out.cpu().numpy(), pix.cpu().numpy()
        return s

    before = state()
    cases = [
        ("null params", lambda: call(None)),
        ("levels 0", lambda: call(prm(levels=0))),
        ("levels 7", lambda: call(prm(levels=7))),
        ("albedo 2", lambda: call(prm(use_albedo=2))),
        ("variance -1", lambda: call(prm(use_variance=-1))),
        ("albedo without preview", lambda: call(prm(use_albedo=1))),
        ("variance without moments", lambda: call(prm(use_variance=1))),
        ("normal_log2 -1", lambda: call(prm(normal_log2=-1))),
        ("normal_log2 9", lambda: call(prm(normal_log2=9))),
        ("sigma_lum < 0", lambda: call(prm(sigma_lum=-1.0))),
        ("sigma_lum nan", lambda: call(prm(sigma_lum=float("nan")))),
        ("sigma_depth 0", lambda: call(prm(sigma_depth=0.0))),
        ("sigma_depth inf", lambda: call(prm(sigma_depth=float("inf")))),
        ("lum_floor 0", lambda: call(prm(lum_floor=0.0))),
        ("lum_floor nan", lambda: call(prm(lum_floor=float("nan")))),
        ("null rgba", lambda: lib.rt_gpu_denoise(hd, C.byref(prm()), None, pp, None)),
        ("host rgba", lambda: call(prm(), o=host.ctypes.data)),
        ("misaligned rgba", lambda: call(prm(), o=op + 4)),
        ("misaligned argb", lambda: call(prm(), a=pp + 2)),
        ("host argb", lambda: call(prm(), a=host.ctypes.data)),
    ]
    for name, fn in cases:
        launches = ctx.launch_count
        assert fn() == rt._abi.RT_ERR_INVALID, name
        assert ctx.launch_count == launches, name
    torch.cuda.synchronize()
    after = state()
    for k in before:
        assert np.array_equal(after[k].view(np.uint8), before[k].view(np.uint8)), k
    # a resize drops the guides (and the readback says so)
    ctx.reset_accum(w + 8, h)
    assert call(prm()) == rt._abi.RT_ERR_INVALID
    assert lib.rt_gpu_readback(hd, rt.RT_READ_GUIDE_NORMAL_F32, host.ctypes.data, host.nbytes) == rt._abi.RT_ERR_NO_SCENE
    with pytest.raises(ValueError):
        ctx.denoise(out=out)                                   # (H, W) of the old size
    # a valid call still works, and counts its launches: the level-0 kernel and one per level
    ctx.render_tile(params(rt, w + 8, h, mode=GUIDES))
    launches = ctx.launch_count
    ctx.denoise(levels=3)
    assert ctx.launch_count == launches + 4
    ctx.synchronize()
    ctx.close()
