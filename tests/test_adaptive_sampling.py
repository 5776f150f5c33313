"""Adaptive sampling: per-pixel moments (rt_gpu_track_moments), renders restricted to a device pixel mask
(rt_gpu_render_masked, GpuContext.render_tile(params, camera, mask)), pixel selection from the error estimate
(rt_gpu_select_pixels) and GpuContext.render_adaptive.

A pixel's samples are keyed by (seed, pixel, pass), so every result is held to render_tile, which the render tests pin
to the reference: a masked pixel equals render_tile's pixel for the same passes, bit for bit, and every other pixel of
every frame buffer keeps its bytes.  Moments and selection are held to float32 numpy restatements of the rules in
include/rt_gpu.h, over per-pass colours taken from single-pass render_tile calls."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import scenes
from conftest import ROOT, bits, same_bits

PATH, PREVIEW, WHITTED, PRIMARY = 0, 1, 2, 3
EXACT, CULLED = 0, 1
W, H = 160, 120
ALL_COUNTERS = ("rays", "camera_rays", "shadow_rays", "node_tests", "tri_tests", "node_visits", "tri_visits", "mesh_hits",
                "mesh_walks")
# under the culled walk the visit counts depend on how packets form
STABLE_COUNTERS = ("rays", "camera_rays", "shadow_rays", "mesh_hits", "mesh_walks")
F32 = np.float32


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
def scene_of(rt, name, data_dir):
    sc = rt.Scene(getattr(scenes, name)(data_dir))
    sc.set_unit_vectors(seed=0, count=1 << 18)
    return sc


def turned_camera(rt, sc):
    d = sc.desc.contents
    lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
    for i in range(d.num_shapes):
        s = d.shapes[i]
        if s.type == 3:
            lo, hi = np.minimum(lo, list(s.bounds_min)), np.maximum(hi, list(s.bounds_max))
    c, h = (lo + hi) / 2, (hi - lo) / 2
    r = float(np.linalg.norm(h)) * 1.3 + 0.2
    return rt.look_at(c + r * np.array([np.sin(2.0), 0.35, np.cos(2.0)]), c)


def dev(a, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a if dtype is None else a.astype(dtype)))
    return t.to("cuda:0")


def region_mask(p):
    """the pixels of [start, end] that the tile fields own, (H, W) bool"""
    pix = np.arange(p.width * p.height)
    x, y = pix % p.width, pix // p.width
    m = (pix >= p.start) & (pix <= p.end)
    if p.tile_count > 1:
        tiles_x = (p.width + p.tile_size - 1) // p.tile_size
        m &= ((y // p.tile_size) * tiles_x + x // p.tile_size) % p.tile_count == p.tile_rank
    return m.reshape(p.height, p.width)


def params(rt, **kw):
    base = dict(mode=PATH, max_bounce=6, antialias=1, seed=3, traverse=CULLED)
    base.update(kw)
    return rt.make_params(base.pop("width", W), base.pop("height", H), **base)


def read_all(rt, ctx, w=W, h=H, preview=False):
    reads = dict(accum=rt.RT_READ_ACCUM_RGBN_F32, display=rt.RT_READ_DISPLAY_ARGB8, ids=rt.RT_READ_PRIMARY_IDS_I32X2,
                 dist=rt.RT_READ_PRIMARY_DIST_F32)
    if preview:
        reads["preview"] = rt.RT_READ_PREVIEW_RGBA_F32
    out = {k: ctx.readback(v, w, h).copy() for k, v in reads.items()}
    out["counters"] = ctx.counters()
    return out


def fresh(ctx, w=W, h=H):
    ctx.reset_accum(w, h)
    ctx.reset_counters()
    ctx.synchronize()


def pass_colours(rt, ctx, p, passes):
    """the pass colour x of every pixel for each pass: single-pass render_tile calls on a reset frame (0 + x = x)"""
    out = []
    for k in passes:
        fresh(ctx, p.width, p.height)
        q = rt._abi.rt_render_params.from_buffer_copy(p)
        q.pass_begin, q.pass_count = k, 1
        ctx.render_tile(q)
        out.append(ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, p.width, p.height)[..., :3].copy())
    return out


def fold_restatement(colours, selected, acc0=None, track=None):
    """accum and moments after folding colours[k] into the pixels selected[k] (bool (H, W)), in order, in float32 with one
    rounding per operation: the fold and the Welford rule of include/rt_gpu.h.  track[k]: moments on for pass k."""
    shape = colours[0].shape[:2]
    s = np.zeros(shape + (3,), F32) if acc0 is None else acc0[..., :3].copy()
    n = np.zeros(shape, np.int64) if acc0 is None else acc0[..., 3].astype(np.int64)
    m2 = np.zeros(shape + (3,), F32)
    w = np.zeros(shape, F32)
    with np.errstate(all="ignore"):
        for k, (x, sel) in enumerate(zip(colours, selected)):
            s1 = (s + x).astype(F32)
            if track is None or track[k]:
                upd = sel & (n > 0)
                n0, n1 = n.astype(F32)[..., None], (n + 1).astype(F32)[..., None]
                d = ((x - s / n0).astype(F32) * (x - s1 / n1).astype(F32)).astype(F32)
                m2 = np.where(upd[..., None], (m2 + d).astype(F32), m2)
                w = np.where(sel, (w + F32(1)).astype(F32), w)
            s = np.where(sel[..., None], s1, s)
            n = n + sel
    return np.concatenate([s, n.astype(F32)[..., None]], -1), np.concatenate([m2, w[..., None]], -1)


def select_restatement(acc, mom, region, mn, mx, abs_tol, rel_tol):
    n = acc[..., 3].astype(np.int64)
    with np.errstate(all="ignore"):
        fn, fn1 = n.astype(F32), (n - 1).astype(F32)
        se = np.sqrt(((mom[..., :3] / fn1[..., None]).astype(F32) / fn[..., None]).astype(F32)).astype(F32)
        mean = (acc[..., :3] / fn[..., None]).astype(F32)
        lum = ((F32(0.2126) * mean[..., 0] + F32(0.7152) * mean[..., 1]).astype(F32) + F32(0.0722) * mean[..., 2]).astype(F32)
        tol = (F32(abs_tol) + F32(rel_tol) * lum).astype(F32)
        over = (se > tol[..., None]).any(-1)
    sel = (n < mx) & ((n < mn) | (mom[..., 3] != fn) | over)
    return (sel & region).astype(np.uint8)


# ---------------------------------------------------------------------------------------------------
# no GPU: layout and bindings
# ---------------------------------------------------------------------------------------------------
def test_select_params_layout_matches_c(rt):
    fields = ("min_passes", "max_passes", "abs_tol", "rel_tol")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rt_gpu.h\"\nint main(void) {\n"
    src += '  printf("size %zu\\n", sizeof(rt_select_params));\n'
    src += '  printf("moments %d\\n", (int)RT_READ_MOMENTS_F32);\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_select_params, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "q.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "q")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    sp = rt._abi.rt_select_params
    assert C.sizeof(sp) == out["size"] == 16
    for f in fields:
        assert getattr(sp, f).offset == out[f], f
    assert rt.RT_READ_MOMENTS_F32 == out["moments"] == 6


def test_adaptive_calls_are_bound(rt):
    lib = rt.load_library()
    for name in ("rt_gpu_track_moments", "rt_gpu_render_masked", "rt_gpu_select_pixels"):
        assert name in rt._abi.GPU_PROTOTYPES
        assert getattr(lib, name).restype is C.c_int
    assert lib.rt_gpu_select_pixels.argtypes[2] is C.POINTER(rt._abi.rt_select_params)


# ---------------------------------------------------------------------------------------------------
# 1. an all-ones mask is render_tile
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_all_ones_mask_is_render_tile(rt, gpu, data_dir):
    import torch
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    cam = turned_camera(rt, sc)
    ones = torch.ones((H, W), dtype=torch.uint8, device="cuda:0")
    tasks = dict(full={}, sub_range=dict(start=W * 17 + 5, end=W * 93 + 130), tiles=dict(tile_size=16, tile_count=3, tile_rank=1))
    for mode in (PATH, PREVIEW, WHITTED, PRIMARY):
        for aa in (0, 1):
            for tr in (EXACT, CULLED):
                for tname, tkw in tasks.items():
                    for c in (None, cam):
                        p = params(rt, mode=mode, antialias=aa, traverse=tr, pass_begin=1, pass_count=2, **tkw)
                        fresh(gpu)
                        gpu.render_tile(p, c)
                        want = read_all(rt, gpu, preview=mode == PREVIEW)
                        fresh(gpu)
                        gpu.render_tile(p, c, mask=ones)
                        got = read_all(rt, gpu, preview=mode == PREVIEW)
                        where = (mode, aa, tr, tname, c is not None)
                        for k in want:
                            if k != "counters":
                                assert same_bits(got[k].view(np.float32), want[k].view(np.float32)), (where, k)
                        for k in (ALL_COUNTERS if tr == EXACT else STABLE_COUNTERS):
                            assert got["counters"][k] == want["counters"][k], (where, k)
                        assert want["counters"]["camera_rays"] > 0


# ---------------------------------------------------------------------------------------------------
# 2. subset masks on a frame that already holds passes
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_subset_masks(rt, gpu, data_dir):
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    cam = turned_camera(rt, sc)
    rng = np.random.default_rng(7)
    rect = np.zeros((H, W), np.uint8)
    rect[30:90, 40:125] = 1
    masks = dict(random30=(rng.random((H, W)) < 0.3).astype(np.uint8), rect=rect, empty=np.zeros((H, W), np.uint8))
    tasks = dict(full={}, sub_tiles=dict(start=W * 11 + 3, end=W * 101 + 7, tile_size=8, tile_count=3, tile_rank=2))
    for mode in (PATH, PREVIEW, WHITTED, PRIMARY):
        for tname, tkw in tasks.items():
            before_p = params(rt, mode=mode, pass_begin=0, pass_count=2)
            p = params(rt, mode=mode, pass_begin=2, pass_count=2, **tkw)
            # render_tile: the same passes on every pixel of the task
            fresh(gpu)
            gpu.render_tile(before_p)
            gpu.synchronize()
            gpu.render_tile(p, cam)
            full = read_all(rt, gpu, preview=mode == PREVIEW)
            region = region_mask(p)
            for mname, m in masks.items():
                fresh(gpu)
                gpu.render_tile(before_p)
                before = read_all(rt, gpu, preview=mode == PREVIEW)
                gpu.reset_counters()
                gpu.render_tile(p, cam, mask=dev(m))
                got = read_all(rt, gpu, preview=mode == PREVIEW)
                sel = region & (m != 0)
                where = (mode, tname, mname)
                for k in before:
                    if k == "counters":
                        continue
                    want = np.where(sel.reshape(sel.shape + (1,) * (got[k].ndim - 2)), full[k], before[k])
                    assert np.array_equal(got[k].view(np.uint8), want.view(np.uint8)), (where, k)
                spp = 4 if mode != PRIMARY else 1
                passes = 2 if mode != PRIMARY else 1
                assert got["counters"]["camera_rays"] == int(sel.sum()) * passes * spp, where


# ---------------------------------------------------------------------------------------------------
# 3.-4. pass history and moments
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode,aa", [(PATH, 1), (WHITTED, 0)])
def test_pass_history_and_moments(rt, gpu, data_dir, mode, aa):
    sc = scene_of(rt, "default_scene", data_dir)
    gpu.upload_scene(sc)
    w, h = 96, 64
    p = params(rt, width=w, height=h, mode=mode, antialias=aa, seed=11)
    P = 9
    cols = pass_colours(rt, gpu, p, range(P))
    rng = np.random.default_rng(3)
    # rounds of a global pass cursor: (first pass, passes, mask)
    rounds = [(0, 2, np.ones((h, w), bool)), (2, 3, rng.random((h, w)) < 0.6), (5, 1, rng.random((h, w)) < 0.5),
              (6, 3, rng.random((h, w)) < 0.3)]
    # moments turned on from the start, and turned on before the third round
    for on_at in (0, 2):
        fresh(gpu, w, h)
        if on_at == 0:
            gpu.track_moments(True)
        selected, track = [None] * P, [False] * P
        for r, (b, k, m) in enumerate(rounds):
            if r == on_at and on_at > 0:
                gpu.track_moments(True)
            q = rt._abi.rt_render_params.from_buffer_copy(p)
            q.pass_begin, q.pass_count = b, k
            gpu.render_tile(q, mask=dev(m, np.uint8))
            for j in range(b, b + k):
                selected[j], track[j] = m, r >= on_at
        acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h)
        mom = gpu.readback(rt.RT_READ_MOMENTS_F32, w, h)
        want_acc, want_mom = fold_restatement(cols, selected, track=track)
        assert same_bits(acc, want_acc), on_at
        assert same_bits(mom, want_mom), on_at
        if on_at == 0:
            assert np.array_equal(mom[..., 3], acc[..., 3])
        else:
            assert (mom[..., 3] < acc[..., 3]).all()
    # tracking off: the moments stay, renders leave them alone; reset_accum zeroes them only while tracking is on
    gpu.track_moments(False)
    q = rt._abi.rt_render_params.from_buffer_copy(p)
    q.pass_begin, q.pass_count = P, 1
    gpu.render_tile(q)
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_MOMENTS_F32, w, h)), bits(mom))
    gpu.reset_accum(w, h)
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_MOMENTS_F32, w, h)), bits(mom))
    gpu.track_moments(True)
    gpu.render_tile(q)
    gpu.reset_accum(w, h)
    assert not gpu.readback(rt.RT_READ_MOMENTS_F32, w, h).any()
    # PREVIEW and PRIMARY leave them alone, as they leave accum
    gpu.render_tile(q)
    after = gpu.readback(rt.RT_READ_MOMENTS_F32, w, h).copy()
    for other in (PREVIEW, PRIMARY):
        gpu.render_tile(params(rt, width=w, height=h, mode=other, pass_begin=1, pass_count=1))
        assert np.array_equal(bits(gpu.readback(rt.RT_READ_MOMENTS_F32, w, h)), bits(after)), other
    # a resize reallocates them, zeroed
    gpu.reset_accum(w + 8, h)
    assert gpu.readback(rt.RT_READ_MOMENTS_F32, w + 8, h).shape == (h, w + 8, 4)
    assert not gpu.readback(rt.RT_READ_MOMENTS_F32, w + 8, h).any()
    gpu.track_moments(False)


# ---------------------------------------------------------------------------------------------------
# 5. selection
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_selection(rt, gpu, data_dir):
    import torch
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    p = params(rt, seed=5)
    full = params(rt)
    rng = np.random.default_rng(1)
    # a frame whose pixels hold different numbers of passes, with NaN sums in some and moments that cover fewer passes
    # than Num in others
    fresh(gpu)
    acc0 = np.zeros((H, W, 4), np.float32)
    acc0[..., 3] = rng.integers(0, 3, (H, W))
    nan_px = rng.random((H, W)) < 0.02
    acc0[nan_px, 0] = np.nan
    acc0[nan_px, 3] = 0
    buf = dev(acc0)
    torch.cuda.synchronize()
    gpu.unpack_owned(full, 0, buf.data_ptr(), buf.numel() * 4)
    gpu.track_moments(True)
    for b, k, frac in ((0, 3, 1.0), (3, 4, 0.7), (7, 6, 0.4), (13, 3, 0.2)):
        q = rt._abi.rt_render_params.from_buffer_copy(p)
        q.pass_begin, q.pass_count = b, k
        gpu.render_tile(q, mask=dev((rng.random((H, W)) < frac).astype(np.uint8)))
    # pixels whose Num no longer matches their moments
    gpu.track_moments(False)
    gpu.render_tile(params(rt, pass_begin=20, pass_count=1, start=W * 50, end=W * 52 - 1))
    gpu.synchronize()
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy()
    mom = gpu.readback(rt.RT_READ_MOMENTS_F32, W, H).copy()
    assert np.isnan(acc[..., 0]).any() and (mom[..., 3] != acc[..., 3]).any()
    n = acc[..., 3]
    assert len(np.unique(n)) >= 6
    regions = dict(full=full, sub=params(rt, start=W * 20 + 7, end=W * 99 + 3),
                   tiles=params(rt, tile_size=16, tile_count=3, tile_rank=2),
                   sub_tiles=params(rt, start=W * 5, end=W * 70 + 11, tile_size=8, tile_count=2, tile_rank=0))
    crits = [(2, 64, 0.0, 0.0), (4, 64, 1e-3, 0.05), (2, 12, 0.01, 0.1), (6, 8, 0.0, 0.02), (2, 2, 0.0, 0.0),
             (3, 10, 0.05, 0.0), (2, 1000, 1e30, 0.0)]
    for rname, reg in regions.items():
        for mn, mx, at, rt_ in crits:
            mask, count = gpu.select_pixels(reg, mn, mx, at, rt_)
            got = mask.cpu().numpy()
            want = select_restatement(acc, mom, region_mask(reg), mn, mx, at, rt_)
            where = (rname, mn, mx, at, rt_)
            assert np.array_equal(got, want), (where, int((got != want).sum()))
            assert int(count.item()) == int(want.sum()), where
    # each clause selects somewhere in the full frame
    reg = region_mask(full)
    assert select_restatement(acc, mom, reg, 2, 1000, 1e30, 0.0).sum() > 0            # m.w != Num / NaN / Num < 2
    assert select_restatement(acc, mom, reg, 2, 64, 0.0, 0.0).sum() > select_restatement(acc, mom, reg, 2, 64, 1e-3, 0.05).sum()
    assert select_restatement(acc, mom, reg, 2, 12, 0.0, 0.0).sum() < select_restatement(acc, mom, reg, 2, 64, 0.0, 0.0).sum()
    # the frame and the moments are inputs only
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(acc))
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_MOMENTS_F32, W, H)), bits(mom))


# ---------------------------------------------------------------------------------------------------
# 6. determinism across scheduling: tiled ranks on frame slots, one pipe, default pipes
# ---------------------------------------------------------------------------------------------------
def adaptive_rounds(rt, ctx, plist, slots, mn, mx, ppr, at, rt_):
    """render_adaptive's loop, interleaved over several regions on several frame slots of one context"""
    for p, s in zip(plist, slots):
        ctx.set_frame_slot(s)
        ctx.reset_accum(p.width, p.height)
        ctx.track_moments(True)
        q = rt._abi.rt_render_params.from_buffer_copy(p)
        q.pass_count = mn
        ctx.render_tile(q)
    cursor, live = mn, list(range(len(plist)))
    while cursor < mx and live:
        sel = {}
        for i in live:
            ctx.set_frame_slot(slots[i])
            sel[i] = ctx.select_pixels(plist[i], mn, mx, at, rt_)
        k = min(ppr, mx - cursor)
        for i in list(live):
            mask, count = sel[i]
            if int(count.item()) == 0:
                live.remove(i)
                continue
            ctx.set_frame_slot(slots[i])
            q = rt._abi.rt_render_params.from_buffer_copy(plist[i])
            q.pass_begin, q.pass_count = plist[i].pass_begin + cursor, k
            ctx.render_tile(q, mask=mask)
        cursor += k
    out = []
    for p, s in zip(plist, slots):
        ctx.set_frame_slot(s)
        out.append((ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, p.width, p.height).copy(),
                    ctx.readback(rt.RT_READ_MOMENTS_F32, p.width, p.height).copy()))
        ctx.track_moments(False)
    ctx.set_frame_slot(0)
    return out


@pytest.mark.gpu
def test_determinism_across_scheduling(rt, data_dir):
    sc = scene_of(rt, "c3_unitychan", data_dir)
    kw = dict(pass_begin=2, seed=9)
    crit = (3, 15, 4, 4e-3, 0.05)
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)
    stats = ctx.render_adaptive(params(rt, **kw), None, *crit)
    acc_default = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy()
    mom_default = ctx.readback(rt.RT_READ_MOMENTS_F32, W, H).copy()
    assert stats["rounds"] >= 2
    assert 3 <= acc_default[..., 3].min() < acc_default[..., 3].max() == 15
    (acc_loop, mom_loop), = adaptive_rounds(rt, ctx, [params(rt, **kw)], [0], *crit)
    assert same_bits(acc_loop, acc_default) and same_bits(mom_loop, mom_default)
    one = rt.GpuContext(0)
    one.set_pipes(1)
    one.upload_scene(sc)
    one.render_adaptive(params(rt, **kw), None, *crit)
    assert same_bits(one.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H), acc_default)
    assert same_bits(one.readback(rt.RT_READ_MOMENTS_F32, W, H), mom_default)
    one.close()
    ranks = [params(rt, tile_size=16, tile_count=3, tile_rank=r, **kw) for r in range(3)]
    for (acc, mom), p in zip(adaptive_rounds(rt, ctx, ranks, [1, 2, 3], *crit), ranks):
        own = region_mask(p)
        assert same_bits(acc[own], acc_default[own]), p.tile_rank
        assert same_bits(mom[own], mom_default[own]), p.tile_rank
        assert not acc[~own].any()
    ctx.close()


# ---------------------------------------------------------------------------------------------------
# 7. stream ordering: a mask written by torch on a side stream
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mask_from_a_side_stream(rt, gpu, data_dir):
    import torch
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    p = params(rt, pass_count=1)
    fresh(gpu)
    gpu.render_tile(p)
    want = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).copy()
    sel = np.zeros((H, W), bool)
    sel[::3, 1::2] = True
    side = torch.cuda.Stream(device=0)
    mask = torch.zeros((H, W), dtype=torch.uint8, device="cuda:0")
    src = dev(sel, np.uint8)
    torch.cuda.synchronize()
    fresh(gpu)
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)           # the mask is written long after the call returns
        mask.copy_(src)
        gpu.render_tile(p, mask=mask)
    gpu.synchronize()
    got = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert same_bits(got[sel], want[sel])
    assert not got[~sel].any()
    # selection: its outputs are complete in the side stream's order, its inputs read after the side stream's work
    gpu.track_moments(True)
    gpu.render_tile(params(rt, pass_begin=1, pass_count=3))
    gpu.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)
        m, count = gpu.select_pixels(p, 2, 64, 0.0, 0.0)
        total = m.sum()
    side.synchronize()
    assert int(count.item()) == int(total.item()) > 0
    gpu.track_moments(False)


# ---------------------------------------------------------------------------------------------------
# 8. convergence
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_convergence(rt, gpu, data_dir):
    sc = scene_of(rt, "c3_unitychan", data_dir)
    gpu.upload_scene(sc)
    w, h = 320, 240
    p = params(rt, width=w, height=h, max_bounce=10)
    mn, mx, at, rt_ = 4, 48, 2e-3, 0.02
    fresh(gpu, w, h)
    stats = gpu.render_adaptive(p, None, min_passes=mn, max_passes=mx, passes_per_round=4, abs_tol=at, rel_tol=rt_)
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h)
    mom = gpu.readback(rt.RT_READ_MOMENTS_F32, w, h)
    assert gpu.counters()["camera_rays"] == stats["camera_rays"]
    n = acc[..., 3]
    # every pixel meets the tolerance or is at max_passes
    left = select_restatement(acc, mom, np.ones((h, w), bool), mn, mx, at, rt_)
    assert not left.any()
    mask, count = gpu.select_pixels(p, mn, mx, at, rt_)
    assert int(count.item()) == 0
    assert (n >= mn).all() and (n <= mx).all() and (n == mx).any() and (n < mx).mean() > 0.3
    assert np.array_equal(mom[..., 3], n)
    assert stats["camera_rays"] == int(n.sum()) * 4
    assert stats["camera_rays"] < w * h * mx * 4
    gpu.track_moments(False)


# ---------------------------------------------------------------------------------------------------
# 9. errors: nothing enqueued, nothing changed
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_errors(rt, data_dir):
    import torch
    lib = rt.load_library()
    sc = scene_of(rt, "c3_unitychan", data_dir)
    ctx = rt.GpuContext(0)
    ctx.upload_scene(sc)
    h = ctx.handle
    p = params(rt, pass_count=1)
    fresh(ctx)
    ctx.set_frame_slot(1)
    fresh(ctx)                                    # slot 1: tracking never on
    ctx.set_frame_slot(0)
    ctx.track_moments(True)
    ctx.render_tile(p)
    ctx.synchronize()
    mask = torch.ones((H, W), dtype=torch.uint8, device="cuda:0")
    count = torch.zeros(2, dtype=torch.int32, device="cuda:0")
    host_mask = np.ones((H, W), np.uint8)
    host_count = np.zeros(1, np.int32)
    torch.cuda.synchronize()

    def state():
        s = read_all(rt, ctx)
        s["moments"] = ctx.readback(rt.RT_READ_MOMENTS_F32, W, H).copy()
        return s

    before = state()
    mp = mask.data_ptr()

    def bad(**kw):
        q = params(rt, pass_count=1)
        for k, v in kw.items():
            setattr(q, k, v)
        return q

    sel = lambda mn=2, mx=8, at=0.0, rt_=0.0: rt._abi.rt_select_params(mn, mx, at, rt_)
    cases = [
        ("masked: null mask", lambda: lib.rt_gpu_render_masked(h, C.byref(p), None, None, None)),
        ("masked: host mask", lambda: lib.rt_gpu_render_masked(h, C.byref(p), None, host_mask.ctypes.data, None)),
        ("masked: unknown mode", lambda: lib.rt_gpu_render_masked(h, C.byref(bad(mode=7)), None, mp, None)),
        ("masked: range", lambda: lib.rt_gpu_render_masked(h, C.byref(bad(end=W * H)), None, mp, None)),
        ("masked: tiles", lambda: lib.rt_gpu_render_masked(h, C.byref(bad(tile_count=3, tile_size=16, tile_rank=3)), None, mp, None)),
        ("masked: bounce", lambda: lib.rt_gpu_render_masked(h, C.byref(bad(max_bounce=40)), None, mp, None)),
        ("masked: camera", lambda: lib.rt_gpu_render_masked(h, C.byref(p), C.byref(rt.camera((0, 0, 7), (1, 0, 0), (2, 0, 0), (0, 0, 1))), mp, None)),
        ("masked: nan camera", lambda: lib.rt_gpu_render_masked(h, C.byref(p), C.byref(rt.camera((0, 0, float("nan")), (1, 0, 0), (0, 1, 0), (0, 0, 1))), mp, None)),
        ("select: min < 2", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel(mn=1)), mp, count.data_ptr(), None)),
        ("select: max < min", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel(mn=5, mx=4)), mp, count.data_ptr(), None)),
        ("select: nan tol", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel(at=float("nan"))), mp, count.data_ptr(), None)),
        ("select: inf tol", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel(rt_=float("inf"))), mp, count.data_ptr(), None)),
        ("select: negative tol", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel(at=-1e-3)), mp, count.data_ptr(), None)),
        ("select: size", lambda: lib.rt_gpu_select_pixels(h, C.byref(bad(width=W + 1, end=W * H)), C.byref(sel()), mp, count.data_ptr(), None)),
        ("select: range", lambda: lib.rt_gpu_select_pixels(h, C.byref(bad(end=W * H)), C.byref(sel()), mp, count.data_ptr(), None)),
        ("select: tiles", lambda: lib.rt_gpu_select_pixels(h, C.byref(bad(tile_count=2, tile_size=0)), C.byref(sel()), mp, count.data_ptr(), None)),
        ("select: null mask", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel()), None, count.data_ptr(), None)),
        ("select: null count", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel()), mp, None, None)),
        ("select: host mask", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel()), host_mask.ctypes.data, count.data_ptr(), None)),
        ("select: host count", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel()), mp, host_count.ctypes.data, None)),
        ("select: misaligned count", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel()), mp, count.data_ptr() + 2, None)),
        ("select: null params", lambda: lib.rt_gpu_select_pixels(h, C.byref(p), None, mp, count.data_ptr(), None)),
    ]
    for name, call in cases:
        launches = ctx.launch_count
        assert call() == rt._abi.RT_ERR_INVALID, name
        assert ctx.launch_count == launches, name
    after = state()
    for k in before:
        if k == "counters":
            assert after[k] == before[k]
        else:
            assert np.array_equal(after[k].view(np.uint8), before[k].view(np.uint8)), k
    # a slot on which tracking was never on: no moments to select from or read back
    ctx.set_frame_slot(1)
    launches = ctx.launch_count
    assert lib.rt_gpu_select_pixels(h, C.byref(p), C.byref(sel()), mp, count.data_ptr(), None) == rt._abi.RT_ERR_INVALID
    assert ctx.launch_count == launches
    out = np.zeros((H, W, 4), np.float32)
    assert lib.rt_gpu_readback(h, rt.RT_READ_MOMENTS_F32, out.ctypes.data, out.nbytes) == rt._abi.RT_ERR_NO_SCENE
    ctx.set_frame_slot(0)
    with pytest.raises(ValueError):
        ctx.render_tile(p, mask=torch.ones((H, W + 1), dtype=torch.uint8, device="cuda:0"))
    with pytest.raises(ValueError):
        ctx.render_tile(p, mask=torch.ones((H, W), dtype=torch.int32, device="cuda:0"))
    # a valid call still works afterwards
    ctx.render_tile(params(rt, pass_begin=1, pass_count=1), mask=mask)
    ctx.synchronize()
    assert (ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)[..., 3] == 2).all()
    ctx.close()
