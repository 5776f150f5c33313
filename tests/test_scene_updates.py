"""Scene updates on the device (rt_gpu_update_mesh / rt_gpu_update_shapes, GpuContext.update_mesh / update_shapes).

The bar: after an update every render, query and radiance call returns, bit for bit, what a fresh upload of the same
scene returns, the mesh built by the host layer from the new points (rt_host_add_mesh_arrays) with the uploaded texture
coordinates and texture slots.  The device arrays are compared byte for byte with the host builder's; results are
compared with a second context that holds the fresh upload."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import scenes
from conftest import ROOT, same_bits
from test_ray_queries import pinhole_rays, random_rays, to_dev

W, H = 64, 48


# ---------------------------------------------------------------------------------------------------
# layout of the update struct (no GPU)
# ---------------------------------------------------------------------------------------------------
def test_mesh_update_layout_matches_c(rt):
    fields = ("points", "num_points", "point_idx", "num_tris", "normals", "num_normals", "normal_idx")
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rt_gpu.h"\nint main(void) {\n'
    src += '  printf("size %zu\\n", sizeof(rt_mesh_update));\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_mesh_update, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "u.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "u")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    u = rt._abi.rt_mesh_update
    assert C.sizeof(u) == out["size"]
    for f in fields:
        assert getattr(u, f).offset == out[f], f


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
SCENES = {
    "torusknot": scenes.c1_torusknot,
    "monkey_plane": scenes.c2_monkey,
    "unitychan": scenes.c3_unitychan,
    "default": scenes.default_scene,
}


def make_scene(rt, spec):
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=0, count=1 << 18)
    return sc


def mesh_shape(sc):
    d = sc.desc.contents
    return next(i for i in range(d.num_shapes) if d.shapes[i].type == 3)        # RT_SHAPE_MESH


def deform(points, kind):
    """float32 (P, 3) -> deformed copy.  rigid: rotation + translation; wobble: per-vertex; aniso: a scale that changes
    split axes; degenerate: collapsed and repeated triangles with signed zeros."""
    p = points.astype(np.float64)
    if kind == "rigid":
        a = 0.7
        R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        p = p @ R.T + np.array([0.3, -0.2, 0.1])
    elif kind == "wobble":
        p = p + 0.05 * np.sin(3.0 * p[:, [1, 2, 0]])
    elif kind == "aniso":
        p = p * np.array([0.3, 2.5, 1.7])
    elif kind == "degenerate":
        out = p.astype(np.float32)
        out[::7] = out[0]                             # triangles collapse onto one point or repeat each other
        out[1::11, 0] = np.float32(-0.0)
        out[2::13, 1] = np.float32(0.0)
        out[5::19, 2] = np.float32(-0.0)
        return out
    return p.astype(np.float32)


def fake_normals(points, seed):
    rng = np.random.default_rng(seed)
    return (rng.normal(size=points.shape)).astype(np.float32)


class Expected:
    """The fresh-upload side: the original scene's description with the updated mesh's arrays and shape bounds taken
    from a host scene built by add_mesh_arrays on the new points (uv and texture slots stay the uploaded ones)."""

    def __init__(self, rt, sc, shape, points, normals=None, nidx=None):
        d = sc.desc.contents
        self.mesh = d.shapes[shape].mesh
        dump = sc.mesh_dump(shape)
        pidx = dump["pidx"].reshape(-1, 3)
        host = rt.Scene()
        host.add_mesh_arrays(points, pidx, normals, nidx, material=("diffuse", (1, 1, 1)))
        nodes, tris, shade = host.flat_mesh(0)
        _, _, shade0 = sc.flat_mesh(self.mesh)
        shade = shade.copy()
        for f in ("uv0", "uv1", "uv2", "texture"):
            shade[f] = shade0[f]
        self.nodes, self.tris, self.shade = nodes, tris, shade
        hb = host.desc.contents.shapes[0]
        self.bounds = np.array(list(hb.bounds_min) + list(hb.bounds_max), np.float32)
        root = np.concatenate([nodes[0]["bmin"], nodes[0]["bmax"]]).astype(np.float32)
        self.cull_scale = np.float32(max([np.float32(0.0)] + [abs(v) for v in root]))
        # the description
        A = rt._abi
        self.shapes = (A.rt_shape * d.num_shapes)()
        C.memmove(self.shapes, d.shapes, C.sizeof(self.shapes))
        for c in range(3):
            self.shapes[shape].bounds_min[c] = hb.bounds_min[c]
            self.shapes[shape].bounds_max[c] = hb.bounds_max[c]
        self.meshes = (A.rt_mesh * d.num_meshes)()
        C.memmove(self.meshes, d.meshes, C.sizeof(self.meshes))
        m = self.meshes[self.mesh]
        m.nodes = self.nodes.ctypes.data_as(C.POINTER(A.rt_bvh_node))
        m.tris = self.tris.ctypes.data_as(C.POINTER(A.rt_tri))
        m.shade = self.shade.ctypes.data_as(C.POINTER(A.rt_shade))
        self.desc = A.rt_scene_desc()
        C.memmove(C.byref(self.desc), C.byref(d), C.sizeof(self.desc))
        self.desc.shapes = self.shapes
        self.desc.meshes = self.meshes
        self.keep = (sc, host)

    def patched_nodes(self):
        n = self.nodes.copy()
        N = len(n)
        for k in np.nonzero(n["tri"] < 0)[0]:
            n["tri"][k] = -2 - (n["escape"][k + 1] if k + 1 < N else N)
        return n

    def leaf_shade(self):
        return self.shade[self.tris["index"]]


def update(gpu, shape, points, pidx, normals=None, nidx=None):
    gpu.update_mesh(shape, to_dev(points), to_dev(pidx.astype(np.int32).reshape(-1, 3)),
                    None if normals is None else to_dev(normals), None if nidx is None else to_dev(nidx.reshape(-1, 3)))


def check_arrays(gpu, exp):
    nodes, tris, shade, bounds, scale = gpu.read_mesh(exp.mesh)
    assert nodes.tobytes() == exp.patched_nodes().tobytes()
    assert tris.tobytes() == exp.tris.tobytes()
    assert shade.tobytes() == exp.leaf_shade().tobytes()
    assert bounds.tobytes() == exp.bounds.tobytes()
    assert np.float32(scale).tobytes() == exp.cull_scale.tobytes()


def frame(rt, ctx, mode=0, traverse=1, max_bounce=4):
    ctx.reset_accum(W, H)
    ctx.render_tile(rt.make_params(W, H, mode=mode, max_bounce=max_bounce, pass_count=1, antialias=0, seed=3,
                                   traverse=traverse))
    return ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)


def check_results(rt, got, want, modes=(0, 1, 2)):
    """query_rays (nearest + occlusion, exact-mode counters), radiance_rays and render_tile: bit for bit."""
    import torch
    rays = to_dev(np.concatenate([pinhole_rays(W, H, True), random_rays(4096, 11)]))
    for traverse in (0, 1):
        res = []
        for ctx in (got, want):
            ctx.synchronize()
            ctx.reset_counters()
            near = ctx.query_rays(rays, traverse=traverse)
            occ = ctx.query_rays(rays, any_hit=True, traverse=traverse)
            torch.cuda.synchronize()
            ctx.synchronize()
            res.append((near["shape"].cpu().numpy(), near["tri"].cpu().numpy(), near["hit"].cpu().numpy(),
                        occ.cpu().numpy(), ctx.counters()))
        a, b = res
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1], b[1])
        assert same_bits(a[2], b[2])
        np.testing.assert_array_equal(a[3], b[3])
        if traverse == 0:
            assert a[4] == b[4]
        for mode in modes:
            ra = got.radiance_rays(rays, mode=mode, max_bounce=4, seed=5, traverse=traverse).cpu().numpy()
            rb = want.radiance_rays(rays, mode=mode, max_bounce=4, seed=5, traverse=traverse).cpu().numpy()
            assert same_bits(ra, rb), (mode, traverse)
        assert same_bits(frame(rt, got, traverse=traverse), frame(rt, want, traverse=traverse))


def fresh(rt, desc):
    ctx = rt.GpuContext(0)
    ctx.upload_scene(C.pointer(desc))
    return ctx


# ---------------------------------------------------------------------------------------------------
# 1. arrays, 2. results
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_update_arrays_equal_host_build(rt, data_dir, name):
    sc = make_scene(rt, SCENES[name](data_dir))
    shape = mesh_shape(sc)
    dump = sc.mesh_dump(shape)
    pts0, pidx = dump["points"], dump["pidx"]
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for kind in ("rigid", "wobble", "aniso", "degenerate"):
            pts = deform(pts0, kind)
            for with_normals in (False, True):
                nrm = fake_normals(pts, 1) if with_normals else None
                nidx = pidx if with_normals else None
                exp = Expected(rt, sc, shape, pts, nrm, None if nidx is None else nidx.reshape(-1, 3))
                update(ctx, shape, pts, pidx, nrm, nidx)
                check_arrays(ctx, exp)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_update_results_equal_fresh_upload(rt, data_dir, name):
    sc = make_scene(rt, SCENES[name](data_dir))
    shape = mesh_shape(sc)
    dump = sc.mesh_dump(shape)
    pidx = dump["pidx"]
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for kind, with_normals in (("wobble", False), ("rigid", True)):
            pts = deform(dump["points"], kind)
            nrm = fake_normals(pts, 2) if with_normals else None
            nidx = pidx.reshape(-1, 3) if with_normals else None
            exp = Expected(rt, sc, shape, pts, nrm, nidx)
            update(ctx, shape, pts, pidx, nrm, nidx)
            ref = fresh(rt, exp.desc)
            try:
                check_results(rt, ctx, ref)
            finally:
                ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 3. sequences A -> B -> A -> C
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_update_sequence(rt, data_dir):
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    dump = sc.mesh_dump(0)
    A, pidx = dump["points"], dump["pidx"]
    B, Cc = deform(A, "wobble"), deform(A, "aniso")
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for pts in (B, A, Cc):
            update(ctx, 0, pts, pidx)
            exp = Expected(rt, sc, 0, pts)
            check_arrays(ctx, exp)
            ref = fresh(rt, exp.desc)
            try:
                check_results(rt, ctx, ref, modes=(0,))
            finally:
                ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 4. ordering across frame slots and streams, without host synchronisation
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_update_ordering_between_slots_and_streams(rt, data_dir):
    """Slot 0 renders a frame large enough to be still running when update_mesh returns (checked with an event), so
    the update has to wait for it on the device before it publishes; slot 1 and a query on the side stream, enqueued
    after the update without a host synchronisation, have to see the new geometry."""
    import torch
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    dump = sc.mesh_dump(0)
    pidx = dump["pidx"]
    new = deform(dump["points"], "rigid")
    exp = Expected(rt, sc, 0, new)
    BW, BH = 1920, 1080
    big = rt.make_params(BW, BH, mode=0, max_bounce=6, pass_count=8, antialias=1, seed=3)
    small = rt.make_params(W, H, mode=0, max_bounce=6, pass_count=1, antialias=0, seed=3)

    def render(ctx, p):
        ctx.reset_accum(p.width, p.height)
        ctx.render_tile(p)
        return ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, p.width, p.height)

    old_ref = rt.GpuContext(0)
    new_ref = fresh(rt, exp.desc)
    ctx = rt.GpuContext(0)
    try:
        old_ref.upload_scene(sc)
        want_old = render(old_ref, big)
        want_new = render(new_ref, small)
        rays = to_dev(pinhole_rays(W, H, True))
        want_q = new_ref.query_rays(rays)["shape"].cpu().numpy()
        ctx.upload_scene(sc)
        for s, p in ((0, big), (1, small)):
            ctx.set_frame_slot(s)
            render(ctx, p)                                # warm-up: pools and buffers sized
            ctx.reset_accum(p.width, p.height)
            ctx.synchronize()
        d_pts, d_idx = to_dev(new), to_dev(pidx.reshape(-1, 3))
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        ctx.set_frame_slot(0)
        ctx.render_tile(big)                              # old geometry
        slot0 = torch.cuda.ExternalStream(ctx.stream)
        frame_done = torch.cuda.Event()
        frame_done.record(slot0)
        with torch.cuda.stream(side):
            ctx.update_mesh(0, d_pts, d_idx)
            assert not frame_done.query(), "the slot-0 frame finished before the update was built: make it larger"
            ctx.set_frame_slot(1)
            ctx.render_tile(small)                        # new geometry
            q = ctx.query_rays(rays)
            got_q = q["shape"].cpu().numpy()
        ctx.set_frame_slot(0)
        got_old = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, BW, BH)
        ctx.set_frame_slot(1)
        got_new = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
        assert same_bits(got_old, want_old)
        assert same_bits(got_new, want_new)
        np.testing.assert_array_equal(got_q, want_q)
    finally:
        ctx.close(); old_ref.close(); new_ref.close()


# ---------------------------------------------------------------------------------------------------
# 5. update_shapes
# ---------------------------------------------------------------------------------------------------
def moved(spec):
    out = []
    for s in spec:
        if s[0] == "sphere":
            out.append(("sphere", tuple(c + 0.25 for c in s[1]), s[2] * 1.1, s[3]))
        elif s[0] == "capsule":
            out.append(("capsule", tuple(c - 0.2 for c in s[1]), tuple(c + 0.1 for c in s[2]), s[3], s[4]))
        elif s[0] == "triangle":
            out.append(("triangle", s[1], tuple(c + 0.3 for c in s[2]), s[3], s[4]))
        else:
            out.append(s)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["default", "mix"])
def test_update_shapes_equals_upload_of_moved_scene(rt, data_dir, name):
    spec = scenes.default_scene(data_dir) if name == "default" else scenes.deterministic_mix(data_dir)
    sc, sc2 = make_scene(rt, spec), make_scene(rt, moved(spec))
    ctx, ref = rt.GpuContext(0), rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        ref.upload_scene(sc2)
        ctx.update_shapes(sc2)
        check_results(rt, ctx, ref, modes=(0, 2))
        # a mesh record's bounds are not taken
        d = sc2.desc.contents
        recs = (rt._abi.rt_shape * d.num_shapes)()
        C.memmove(recs, d.shapes, C.sizeof(recs))
        mi = mesh_shape(sc2)
        recs[mi].bounds_min[0] = -1e30
        recs[mi].bounds_max[1] = 1e30
        ctx._check(ctx._lib.rt_gpu_update_shapes(ctx.handle, recs, 0, d.num_shapes, None))
        check_results(rt, ctx, ref, modes=(0,))
        # type, mesh and has_bounds stay those of the upload
        for field, value in (("type", 0 if recs[0].type != 0 else 2), ("mesh", 0), ("has_bounds", 1 - recs[0].has_bounds)):
            bad = (rt._abi.rt_shape * 1)()
            C.memmove(bad, recs, C.sizeof(bad))
            setattr(bad[0], field, value)
            assert ctx._lib.rt_gpu_update_shapes(ctx.handle, bad, 0, 1, None) == rt._abi.RT_ERR_INVALID, field
        bad = (rt._abi.rt_shape * 1)()
        C.memmove(bad, recs, C.sizeof(bad))
        bad[0].material = 10_000
        assert ctx._lib.rt_gpu_update_shapes(ctx.handle, bad, 0, 1, None) == rt._abi.RT_ERR_INVALID
        assert ctx._lib.rt_gpu_update_shapes(ctx.handle, recs, d.num_shapes - 1, 2, None) == rt._abi.RT_ERR_INVALID
        check_results(rt, ctx, ref, modes=(0,))
    finally:
        ctx.close(); ref.close()


# ---------------------------------------------------------------------------------------------------
# 6. errors leave the scene as it was
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_update_errors_leave_the_scene(rt, data_dir):
    import torch
    A = rt._abi
    sc = make_scene(rt, scenes.deterministic_mix(data_dir))
    shape = mesh_shape(sc)
    dump = sc.mesh_dump(shape)
    pts, pidx = deform(dump["points"], "wobble"), dump["pidx"].reshape(-1, 3).astype(np.int32)
    T = len(pidx)
    ctx = rt.GpuContext(0)
    try:
        u = A.rt_mesh_update()
        assert ctx._lib.rt_gpu_update_mesh(ctx.handle, shape, C.byref(u), None) == A.RT_ERR_NO_SCENE
        ctx.upload_scene(sc)
        before = frame(rt, ctx)
        d_pts, d_idx = to_dev(pts), to_dev(pidx)
        d_nrm = to_dev(fake_normals(pts, 3))

        def call(shape=shape, points=d_pts.data_ptr(), num_points=len(pts), point_idx=d_idx.data_ptr(), num_tris=T,
                 normals=None, num_normals=0, normal_idx=None):
            u = A.rt_mesh_update(points, num_points, point_idx, num_tris, normals, num_normals, normal_idx)
            return ctx._lib.rt_gpu_update_mesh(ctx.handle, shape, C.byref(u), None)

        host_pts = np.ascontiguousarray(pts)
        bad_idx = pidx.copy(); bad_idx[T // 2, 1] = len(pts)
        neg_idx = pidx.copy(); neg_idx[T - 1, 2] = -1
        bad_nidx = pidx.copy(); bad_nidx[3, 0] = len(pts)
        d_bad, d_neg, d_bad_n = to_dev(bad_idx), to_dev(neg_idx), to_dev(bad_nidx)
        torch.cuda.synchronize()
        cases = [
            dict(points=None), dict(point_idx=None),
            dict(points=d_pts.data_ptr() + 2),                       # misaligned
            dict(points=host_pts.ctypes.data),                       # host memory
            dict(shape=0),                                           # a sphere
            dict(shape=-1), dict(shape=10_000),
            dict(num_tris=T - 1), dict(num_points=0),
            dict(normals=d_nrm.data_ptr(), num_normals=len(pts)),    # normals without normal_idx
            dict(normal_idx=d_idx.data_ptr()),                       # and the reverse
            dict(point_idx=d_bad.data_ptr()), dict(point_idx=d_neg.data_ptr()),     # found on the device
            dict(normals=d_nrm.data_ptr(), num_normals=len(pts), normal_idx=d_bad_n.data_ptr()),
        ]
        for kw in cases:
            assert call(**kw) == A.RT_ERR_INVALID, kw
            assert same_bits(frame(rt, ctx), before), kw
        # a mesh that two shapes reference is rejected
        d = sc.desc.contents
        shapes = (A.rt_shape * (d.num_shapes + 1))()
        C.memmove(shapes, d.shapes, C.sizeof(A.rt_shape) * d.num_shapes)
        shapes[d.num_shapes] = shapes[shape]
        desc2 = A.rt_scene_desc()
        C.memmove(C.byref(desc2), C.byref(d), C.sizeof(desc2))
        desc2.shapes, desc2.num_shapes = shapes, d.num_shapes + 1
        ctx2 = rt.GpuContext(0)
        try:
            ctx2.upload_scene(C.pointer(desc2))
            u = A.rt_mesh_update(d_pts.data_ptr(), len(pts), d_idx.data_ptr(), T, None, 0, None)
            assert ctx2._lib.rt_gpu_update_mesh(ctx2.handle, shape, C.byref(u), None) == A.RT_ERR_INVALID
        finally:
            ctx2.close()
        # the torch layer
        for args in ((d_pts.cpu(), d_idx), (d_pts.double(), d_idx), (d_pts, d_idx.long()), (d_pts[:, :2], d_idx),
                     (d_pts, d_idx, d_nrm, None), (d_pts, d_idx, None, d_idx), (d_pts, d_idx.t()),
                     (d_pts, d_idx, d_nrm, d_idx[:-1])):
            with pytest.raises(ValueError):
                ctx.update_mesh(shape, *args)
        with pytest.raises(rt.RtError):
            ctx.update_mesh(shape, d_pts, d_bad)
        assert same_bits(frame(rt, ctx), before)
        # and a valid update still works afterwards
        ctx.update_mesh(shape, d_pts, d_idx)
        exp = Expected(rt, sc, shape, pts)
        check_arrays(ctx, exp)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_update_rejects_a_mesh_whose_nodes_are_not_its_tree(rt, data_dir):
    """A description may carry a node array of another size than 2T-1 (a forest after the root, or a tree over some of
    the triangles): an update would publish 2T-1 nodes under the uploaded count, so it is refused."""
    A = rt._abi
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    dump = sc.mesh_dump(0)
    pts, pidx = deform(dump["points"], "wobble"), dump["pidx"].reshape(-1, 3).astype(np.int32)
    nodes, tris, shade = sc.flat_mesh(0)
    N = len(nodes)
    extra = np.zeros(1, nodes.dtype)                      # a one-leaf tree after the root's escape
    extra["bmin"], extra["bmax"], extra["escape"], extra["tri"] = nodes[1]["bmin"], nodes[1]["bmax"], N + 1, 0
    longer = np.concatenate([nodes, extra])
    leaf = np.zeros(1, nodes.dtype)                       # a tree of triangle 0 alone
    leaf["bmin"], leaf["bmax"], leaf["escape"], leaf["tri"] = nodes[0]["bmin"], nodes[0]["bmax"], 1, 0
    d_pts, d_idx = to_dev(pts), to_dev(pidx)
    import torch
    torch.cuda.synchronize()
    for arr in (longer, leaf):
        d = sc.desc.contents
        meshes = (A.rt_mesh * d.num_meshes)()
        C.memmove(meshes, d.meshes, C.sizeof(meshes))
        meshes[0].nodes = arr.ctypes.data_as(C.POINTER(A.rt_bvh_node))
        meshes[0].num_nodes = len(arr)
        desc = A.rt_scene_desc()
        C.memmove(C.byref(desc), C.byref(d), C.sizeof(desc))
        desc.meshes = meshes
        ctx = rt.GpuContext(0)
        try:
            ctx.upload_scene(C.pointer(desc))
            before = frame(rt, ctx)
            u = A.rt_mesh_update(d_pts.data_ptr(), len(pts), d_idx.data_ptr(), len(pidx), None, 0, None)
            assert ctx._lib.rt_gpu_update_mesh(ctx.handle, 0, C.byref(u), None) == A.RT_ERR_INVALID, len(arr)
            with pytest.raises(rt.RtError):
                ctx.update_mesh(0, d_pts, d_idx)
            assert same_bits(frame(rt, ctx), before)
            got_nodes = ctx.read_mesh(0)[0]                # the uploaded array, whole
            np.testing.assert_array_equal(got_nodes["escape"], arr["escape"])
        finally:
            ctx.close()


@pytest.mark.gpu
def test_update_shapes_many_records(rt, data_dir):
    """More records than one launch carries: 130 spheres moved at once equal an upload of the moved scene."""
    rng = np.random.default_rng(4)
    spec = [("sphere", tuple(map(float, rng.uniform(-3, 3, 3) - [0, 0, 3])), float(rng.uniform(0.1, 0.4)),
             ("reflective", (0.8, 0.7, 0.6), 0.0)) for _ in range(130)]
    spec.append(("mesh", os.path.join(data_dir, "TorusKnot.obj"), ("reflective", (0.8, 0.6, 0.4), 0.0)))
    sc, sc2 = make_scene(rt, spec), make_scene(rt, moved(spec))
    ctx, ref = rt.GpuContext(0), rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        ref.upload_scene(sc2)
        ctx.update_shapes(sc2, first=3, count=len(spec) - 3)
        ctx.update_shapes(sc2, first=0, count=3)
        check_results(rt, ctx, ref, modes=(0, 2))
    finally:
        ctx.close(); ref.close()
