"""Mesh replacement on the device (rt_gpu_replace_mesh, GpuContext.replace_mesh): new geometry of any triangle count,
with texture coordinates and texture slots, from device memory.

The bar: after a replace every render, query and radiance call returns, bit for bit, what a fresh upload returns of
the scene in which the mesh is rt_host_add_mesh_arrays(points, normals, texcoords, point_idx, normal_idx, texcoord_idx)
with shade[t].texture = texture[t] and the mesh's uploaded texture slots.  The device arrays are compared byte for byte
with that host build; results are compared with a second context that holds the fresh upload."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import scenes
from conftest import ROOT, same_bits
from test_ray_queries import pinhole_rays, to_dev
from test_scene_refit import refit_reference
from test_scene_updates import Expected, check_arrays, check_results, deform, fake_normals, fresh, make_scene

F32 = np.float32
W, H = 64, 48


# ---------------------------------------------------------------------------------------------------
# no GPU: the struct's layout, and the comparator pinned to the loader
# ---------------------------------------------------------------------------------------------------
def test_mesh_replace_layout_matches_c(rt):
    fields = ("geometry", "texcoords", "num_texcoords", "texcoord_idx", "texture")
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rt_gpu.h"\nint main(void) {\n'
    src += '  printf("size %zu\\n", sizeof(rt_mesh_replace));\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_mesh_replace, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "r.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "r")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    r = rt._abi.rt_mesh_replace
    assert C.sizeof(r) == out["size"]
    for f in fields:
        assert getattr(r, f).offset == out[f], f


class ReplaceExpected(Expected):
    """The fresh-upload side of a replace: the original scene's description with the mesh's arrays, counts and shape
    bounds taken from a host scene built by add_mesh_arrays on the new arrays, the texture slots patched in."""

    def __init__(self, rt, sc, shape, g):
        d = sc.desc.contents
        self.mesh = d.shapes[shape].mesh
        host = rt.Scene()
        host.add_mesh_arrays(g["points"], g["pidx"], g.get("normals"), g.get("nidx"), g.get("texcoords"), g.get("tidx"),
                             material=("diffuse", (1, 1, 1)))
        nodes, tris, shade = host.flat_mesh(0)
        shade = shade.copy()
        if g.get("texture") is not None:
            shade["texture"] = np.asarray(g["texture"], np.int32)
        self.nodes, self.tris, self.shade = nodes, tris, shade
        hb = host.desc.contents.shapes[0]
        self.bounds = np.array(list(hb.bounds_min) + list(hb.bounds_max), F32)
        self._set_scale()
        A = rt._abi
        self.shapes = (A.rt_shape * d.num_shapes)()
        C.memmove(self.shapes, d.shapes, C.sizeof(self.shapes))
        for c in range(3):
            self.shapes[shape].bounds_min[c] = hb.bounds_min[c]
            self.shapes[shape].bounds_max[c] = hb.bounds_max[c]
        self.meshes = (A.rt_mesh * d.num_meshes)()
        C.memmove(self.meshes, d.meshes, C.sizeof(self.meshes))
        self._set_arrays(A)
        self.desc = A.rt_scene_desc()
        C.memmove(C.byref(self.desc), C.byref(d), C.sizeof(self.desc))
        self.desc.shapes = self.shapes
        self.desc.meshes = self.meshes
        self.keep = (sc, host)

    def _set_scale(self):
        root = np.concatenate([self.nodes[0]["bmin"], self.nodes[0]["bmax"]]).astype(F32)
        self.cull_scale = F32(max([F32(0.0)] + [abs(v) for v in root]))

    def _set_arrays(self, A):
        m = self.meshes[self.mesh]
        m.nodes = self.nodes.ctypes.data_as(C.POINTER(A.rt_bvh_node))
        m.tris = self.tris.ctypes.data_as(C.POINTER(A.rt_tri))
        m.shade = self.shade.ctypes.data_as(C.POINTER(A.rt_shade))
        m.num_nodes, m.num_tris = len(self.nodes), len(self.tris)

    def refit(self, rt, points):
        """The same mesh after a refit to `points`: the topology of these arrays, shading from the new points."""
        g = dict(self.g, points=points)
        g.pop("normals", None), g.pop("nidx", None)          # refit_mesh is called without normals
        exp = ReplaceExpected.make(rt, self.keep[0], self.shape, g)
        exp.nodes, exp.tris = refit_reference(self.nodes, self.tris, points, g["pidx"])
        exp._set_scale()
        exp._set_arrays(rt._abi)
        return exp

    @classmethod
    def make(cls, rt, sc, shape, g):
        exp = cls(rt, sc, shape, g)
        exp.g, exp.shape = g, shape
        return exp


def test_replace_comparator_is_the_loader(rt, data_dir):
    """add_mesh_arrays fed a loaded textured mesh's own arrays, with the loaded texture slots patched in, gives the
    loaded mesh's flat nodes, triangles and shading records byte for byte: the expected side is the host layer's."""
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    d = sc.mesh_dump(0)
    nodes, tris, shade = sc.flat_mesh(0)
    assert (shade["texture"] >= 0).any()
    exp = ReplaceExpected(rt, sc, 0, dict(points=d["points"], pidx=d["pidx"].reshape(-1, 3), normals=d["normals"],
                                          nidx=d["nidx"].reshape(-1, 3), texcoords=d["texcoords"][:, :2],
                                          tidx=d["tidx"].reshape(-1, 3), texture=shade["texture"]))
    assert exp.nodes.tobytes() == nodes.tobytes()
    assert exp.tris.tobytes() == tris.tobytes()
    assert exp.shade.tobytes() == shade.tobytes()


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
def grid(n, seed=0):
    """A parametric height field of 2 n^2 triangles around the origin, facing the camera, with uv per point."""
    u = np.linspace(-1.6, 1.6, n + 1).astype(F32)
    X, Y = np.meshgrid(u, u)
    Z = (0.3 * np.sin(3.0 * X + seed) * np.cos(2.0 * Y + 0.5 * seed)).astype(F32)
    pts = np.stack([X, Y, Z], -1).reshape(-1, 3).astype(F32)
    a = (np.arange(n)[:, None] * (n + 1) + np.arange(n)[None, :]).ravel()
    b, c = a + 1, a + n + 1
    pidx = np.stack([np.stack([a, b, c + 1], 1), np.stack([a, c + 1, c], 1)], 1).reshape(-1, 3).astype(np.int32)
    uv = np.stack([(X.ravel() + 1.6) / 3.2, (Y.ravel() + 1.6) / 3.2], 1).astype(F32)
    return dict(points=pts, pidx=pidx, texcoords=uv, tidx=pidx.copy())


def geometry(g, normals=False, texcoords=False, slots=None, seed=1):
    """g with or without normals (random, indexed like the points) and texcoords, and texture slots cycling `slots`."""
    out = dict(points=g["points"], pidx=g["pidx"])
    if normals:
        out["normals"], out["nidx"] = fake_normals(g["points"], seed), g["pidx"]
    if texcoords:
        out["texcoords"], out["tidx"] = g["texcoords"], g["tidx"]
    if slots is not None:
        out["texture"] = np.resize(np.asarray(slots, np.int32), len(g["pidx"]))
    return out


def replace(ctx, shape, g):
    dev = lambda k, dt=None: None if g.get(k) is None else to_dev(np.ascontiguousarray(g[k], dt))
    ctx.replace_mesh(shape, dev("points", F32), dev("pidx", np.int32), dev("normals", F32), dev("nidx", np.int32),
                     dev("texcoords", F32), dev("tidx", np.int32), dev("texture", np.int32))


def uploaded_geometry(sc, shape):
    """The uploaded mesh's own arrays as a replace takes them (same count, uploaded uv and slots)."""
    d = sc.mesh_dump(shape)
    _, _, shade = sc.flat_mesh(sc.desc.contents.shapes[shape].mesh)
    return dict(points=d["points"], pidx=d["pidx"].reshape(-1, 3), texcoords=d["texcoords"][:, :2].copy(),
                tidx=d["tidx"].reshape(-1, 3), texture=shade["texture"].copy())


def textured_slots(sc, mesh):
    _, _, shade = sc.flat_mesh(mesh)
    return sorted(set(int(s) for s in shade["texture"] if s >= 0))


def mesh_bytes(ctx, mesh):
    return [np.asarray(a).tobytes() for a in ctx.read_mesh(mesh)]


def scene_bytes(ctx):
    return ctx._lib.rt_gpu_scene_bytes(ctx.handle)


def torus_sizes(sc):
    """grid sizes around the uploaded TorusKnot's count T0: a shrink, one between T0 and the grow, and a grow."""
    T0 = len(sc.mesh_dump(0)["pidx"]) // 3
    return 20, int(np.ceil(np.sqrt(T0 / 2))) + 3, int(np.ceil(np.sqrt(T0))) + 10


# ---------------------------------------------------------------------------------------------------
# 1. arrays, 2. results
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_replace_arrays_equal_host_build_torusknot(rt, data_dir):
    """TorusKnot into generated grids: a shrink, a grow past capacity, the same count, a shrink; with and without
    normals and texcoords; negative texture slots pass unchanged."""
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    small, mid, big = torus_sizes(sc)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        steps = [grid(small), grid(big), grid(big, seed=2), grid(mid, seed=3)]
        steps[2]["points"] = deform(steps[2]["points"], "degenerate")
        for k, g in enumerate(steps):
            for normals, texcoords in ((False, False), (True, False), (False, True), (True, True)):
                geo = geometry(g, normals, texcoords, slots=[-1, -7] if texcoords else None, seed=k)
                replace(ctx, 0, geo)
                check_arrays(ctx, ReplaceExpected(rt, sc, 0, geo))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_replace_arrays_equal_host_build_unitychan(rt, data_dir):
    """unitychan with new uv and texture slots cycling over its textured slots and -1, then a grid with its own uv;
    a same-count replace with the uploaded uv and slots gives update_mesh's bytes."""
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    slots = textured_slots(sc, 0) + [-1]
    up = uploaded_geometry(sc, 0)
    rng = np.random.default_rng(5)
    ctx, ref = rt.GpuContext(0), rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        own = dict(up, points=deform(up["points"], "wobble"), texcoords=rng.uniform(-0.5, 1.5, (len(up["points"]), 2)).astype(F32),
                   tidx=up["pidx"], texture=np.resize(np.asarray(slots, np.int32), len(up["pidx"])))
        for geo in (own, dict(own, normals=fake_normals(own["points"], 4), nidx=up["pidx"]),
                    geometry(grid(70), texcoords=True, slots=slots), geometry(grid(30), normals=True, slots=slots[::-1])):
            replace(ctx, 0, geo)
            check_arrays(ctx, ReplaceExpected(rt, sc, 0, geo))
        # the same count with the uploaded uv and slots: update_mesh's arrays
        pts = deform(up["points"], "rigid")
        replace(ctx, 0, dict(up, points=pts))
        ref.upload_scene(sc)
        ref.update_mesh(0, to_dev(pts), to_dev(up["pidx"]))
        assert mesh_bytes(ctx, 0) == mesh_bytes(ref, 0)
        check_arrays(ctx, Expected(rt, sc, 0, pts))
    finally:
        ctx.close(); ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["torusknot", "unitychan", "default"])
def test_replace_results_equal_fresh_upload(rt, data_dir, name):
    spec = {"torusknot": scenes.c1_torusknot, "unitychan": scenes.c3_unitychan, "default": scenes.default_scene}[name](data_dir)
    sc = make_scene(rt, spec)
    d = sc.desc.contents
    shape = next(i for i in range(d.num_shapes) if d.shapes[i].type == rt._abi.RT_SHAPE_MESH)
    slots = textured_slots(sc, d.shapes[shape].mesh) + [-1]
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for geo in (geometry(grid(120), texcoords=True, slots=slots), geometry(grid(25, seed=1), normals=True, slots=slots[1:] or [-1])):
            replace(ctx, shape, geo)
            exp = ReplaceExpected(rt, sc, shape, geo)
            ref = fresh(rt, exp.desc)
            try:
                check_results(rt, ctx, ref)
            finally:
                ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 3. sequences with refits and updates
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_replace_sequence(rt, data_dir):
    """replace (grow), refit, update_mesh, replace (shrink), refit, then replaces alternating between two levels of
    detail; arrays and results after every step."""
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    small, mid, big = torus_sizes(sc)
    hi, lo = geometry(grid(big), texcoords=True, slots=[-1]), geometry(grid(mid, seed=1), normals=True)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        exp = None
        for op, arg in (("replace", hi), ("refit", "wobble"), ("update", "aniso"), ("replace", geometry(grid(small))),
                        ("refit", "rigid"), ("replace", lo), ("replace", hi), ("replace", lo)):
            if op == "replace":
                replace(ctx, 0, arg)
                exp = ReplaceExpected.make(rt, sc, 0, arg)
            elif op == "refit":
                pts = deform(exp.g["points"], arg)
                status = ctx.refit_mesh(0, to_dev(pts), to_dev(exp.g["pidx"]))
                assert status.item() == 0
                exp = exp.refit(rt, pts)
            else:
                g = dict(exp.g, points=deform(exp.g["points"], arg))
                g.pop("normals", None), g.pop("nidx", None)
                ctx.update_mesh(0, to_dev(g["points"]), to_dev(g["pidx"]))
                exp = ReplaceExpected.make(rt, sc, 0, g)
            check_arrays(ctx, exp)
            ref = fresh(rt, exp.desc)
            try:
                check_results(rt, ctx, ref, modes=(0,))
            finally:
                ref.close()
    finally:
        ctx.close()


def with_nodes(rt, sc, nodes):
    """sc's description with mesh 0's node array replaced (kept alive by the returned tuple)."""
    A = rt._abi
    d = sc.desc.contents
    meshes = (A.rt_mesh * d.num_meshes)()
    C.memmove(meshes, d.meshes, C.sizeof(meshes))
    meshes[0].nodes = nodes.ctypes.data_as(C.POINTER(A.rt_bvh_node))
    meshes[0].num_nodes = len(nodes)
    desc = A.rt_scene_desc()
    C.memmove(C.byref(desc), C.byref(d), C.sizeof(desc))
    desc.meshes = meshes
    return desc, (meshes, nodes)


@pytest.mark.gpu
def test_replace_accepts_meshes_update_and_refit_refuse(rt, data_dir):
    """Uploaded node arrays that update_mesh refuses (not 2T-1 nodes) or refit_mesh refuses (a slot named twice): a
    replace publishes a tree of its own, after which both accept the mesh."""
    import torch
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    dump = sc.mesh_dump(0)
    pidx = dump["pidx"].reshape(-1, 3).astype(np.int32)
    nodes, _, _ = sc.flat_mesh(0)
    N = len(nodes)
    extra = np.zeros(1, nodes.dtype)                      # 2T nodes: a one-leaf tree after the root's escape
    extra["bmin"], extra["bmax"], extra["escape"], extra["tri"] = nodes[1]["bmin"], nodes[1]["bmax"], N + 1, 0
    leaf = np.zeros(1, nodes.dtype)                       # one node: a tree of triangle 0 alone
    leaf["bmin"], leaf["bmax"], leaf["escape"], leaf["tri"] = nodes[0]["bmin"], nodes[0]["bmax"], 1, 0
    twice = nodes.copy()                                  # 2T-1 nodes, one leaf slot named twice
    leaves = np.nonzero(twice["tri"] >= 0)[0]
    twice["tri"][leaves[1]] = twice["tri"][leaves[0]]
    g = geometry(grid(40), texcoords=True)
    for arr in (np.concatenate([nodes, extra]), leaf, twice):
        desc, keep = with_nodes(rt, sc, arr)
        ctx = rt.GpuContext(0)
        try:
            ctx.upload_scene(C.pointer(desc))
            d_pts, d_idx = to_dev(dump["points"]), to_dev(pidx)
            torch.cuda.synchronize()
            with pytest.raises(rt.RtError):
                if len(arr) == N:
                    ctx.refit_mesh(0, d_pts, d_idx)
                else:
                    ctx.update_mesh(0, d_pts, d_idx)
            replace(ctx, 0, g)
            check_arrays(ctx, ReplaceExpected(rt, sc, 0, g))
            pts = deform(g["points"], "wobble")
            ctx.update_mesh(0, to_dev(pts), to_dev(g["pidx"]))
            exp = ReplaceExpected.make(rt, sc, 0, dict(g, points=pts))
            check_arrays(ctx, exp)
            pts2 = deform(g["points"], "aniso")
            assert ctx.refit_mesh(0, to_dev(pts2), to_dev(g["pidx"])).item() == 0
            check_arrays(ctx, exp.refit(rt, pts2))
        finally:
            ctx.close()


# ---------------------------------------------------------------------------------------------------
# 4. ordering across frame slots and streams
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_replace_ordering_between_slots_and_streams(rt, data_dir):
    """A slot-0 frame still running when the replace returns sees the old mesh; slot 1 and a query on the side
    stream, enqueued after it without a host synchronisation, see the new one."""
    import torch
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    geo = geometry(grid(60), texcoords=True, slots=textured_slots(sc, 0) + [-1])
    exp = ReplaceExpected(rt, sc, 0, geo)
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
        want_q = new_ref.query_rays(rays)
        want_q = (want_q["shape"].cpu().numpy(), want_q["tri"].cpu().numpy())
        ctx.upload_scene(sc)
        for s, p in ((0, big), (1, small)):
            ctx.set_frame_slot(s)
            render(ctx, p)                                # warm-up: pools and buffers sized
            ctx.reset_accum(p.width, p.height)
            ctx.synchronize()
        d = {k: to_dev(np.ascontiguousarray(v)) for k, v in geo.items()}
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        ctx.set_frame_slot(0)
        ctx.render_tile(big)                              # old mesh
        slot0 = torch.cuda.ExternalStream(ctx.stream)
        frame_done = torch.cuda.Event()
        frame_done.record(slot0)
        with torch.cuda.stream(side):
            ctx.replace_mesh(0, d["points"], d["pidx"], texcoords=d["texcoords"], texcoord_idx=d["tidx"], texture=d["texture"])
            assert not frame_done.query(), "the slot-0 frame finished before the replace returned: make it larger"
            ctx.set_frame_slot(1)
            ctx.render_tile(small)                        # new mesh
            q = ctx.query_rays(rays)
            got_q = (q["shape"].cpu().numpy(), q["tri"].cpu().numpy())
        ctx.set_frame_slot(0)
        got_old = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, BW, BH)
        ctx.set_frame_slot(1)
        got_new = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
        assert same_bits(got_old, want_old)
        assert same_bits(got_new, want_new)
        np.testing.assert_array_equal(got_q[0], want_q[0])
        np.testing.assert_array_equal(got_q[1], want_q[1])
    finally:
        ctx.close(); old_ref.close(); new_ref.close()


# ---------------------------------------------------------------------------------------------------
# 5. errors leave the scene as it was
# ---------------------------------------------------------------------------------------------------
def with_empty_slot(rt, sc):
    """sc's description with one texture slot without pixels appended to mesh 0's textures."""
    A = rt._abi
    d = sc.desc.contents
    meshes = (A.rt_mesh * d.num_meshes)()
    C.memmove(meshes, d.meshes, C.sizeof(meshes))
    n = meshes[0].num_textures
    texs = (A.rt_texture * (n + 1))()
    C.memmove(texs, meshes[0].textures, C.sizeof(A.rt_texture) * n)
    meshes[0].textures, meshes[0].num_textures = texs, n + 1
    desc = A.rt_scene_desc()
    C.memmove(C.byref(desc), C.byref(d), C.sizeof(desc))
    desc.meshes = meshes
    return desc, (meshes, texs), n


@pytest.mark.gpu
def test_replace_errors_leave_the_scene(rt, data_dir):
    """Every host rejection and every bad index or slot found on the device (also in a replace that grows past
    capacity) leaves the arrays byte for byte; a good replace, refit and update follow."""
    import torch
    A = rt._abi
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    desc, keep, empty = with_empty_slot(rt, sc)
    g = geometry(grid(50), normals=True, texcoords=True, slots=textured_slots(sc, 0) + [-1])
    T = len(g["pidx"])
    big = geometry(grid(120), texcoords=True)
    ctx = rt.GpuContext(0)
    try:
        r = A.rt_mesh_replace()
        assert ctx._lib.rt_gpu_replace_mesh(ctx.handle, 0, C.byref(r), None) == A.RT_ERR_NO_SCENE
        ctx.upload_scene(C.pointer(desc))
        d = {k: to_dev(np.ascontiguousarray(v)) for k, v in g.items()}
        db = {k: to_dev(np.ascontiguousarray(v)) for k, v in big.items()}
        host_pts, host_tex = np.ascontiguousarray(g["points"]), np.ascontiguousarray(g["texture"])

        def bad(key, row, col, value, src=g):
            a = np.array(src[key], copy=True)
            if a.ndim == 2:
                a[row, col] = value
            else:
                a[row] = value
            return to_dev(a)

        def call(shape=0, points=d["points"].data_ptr(), num_points=len(g["points"]), point_idx=d["pidx"].data_ptr(),
                 num_tris=T, normals=d["normals"].data_ptr(), num_normals=len(g["normals"]), normal_idx=d["nidx"].data_ptr(),
                 texcoords=d["texcoords"].data_ptr(), num_texcoords=len(g["texcoords"]), texcoord_idx=d["tidx"].data_ptr(),
                 texture=d["texture"].data_ptr()):
            u = A.rt_mesh_update(points, num_points, point_idx, num_tris, normals, num_normals, normal_idx)
            r = A.rt_mesh_replace(u, texcoords, num_texcoords, texcoord_idx, texture)
            return ctx._lib.rt_gpu_replace_mesh(ctx.handle, shape, C.byref(r), None)

        P, Q = len(g["points"]), len(g["texcoords"])
        device_bad = dict(
            point=bad("pidx", T // 2, 1, P), point_neg=bad("pidx", T - 1, 2, -1),
            normal=bad("nidx", 3, 0, P), texcoord=bad("tidx", 7, 2, Q), texcoord_neg=bad("tidx", 0, 0, -1),
            slot=bad("texture", 11, 0, empty + 1), slot_empty=bad("texture", T - 1, 0, empty),
            grow=bad("tidx", len(big["pidx"]) - 1, 1, len(big["texcoords"]), src=big))
        torch.cuda.synchronize()
        for round_ in range(2):                           # before any replace, then with a spare set in place
            before = mesh_bytes(ctx, 0)
            cases = [
                dict(points=None), dict(point_idx=None), dict(shape=-1), dict(shape=10_000), dict(num_tris=0),
                dict(num_tris=-3), dict(num_points=0),
                dict(points=d["points"].data_ptr() + 2), dict(points=host_pts.ctypes.data),
                dict(normal_idx=None), dict(normals=None), dict(num_normals=0),
                dict(texcoord_idx=None), dict(texcoords=None), dict(num_texcoords=0),
                dict(texcoords=d["texcoords"].data_ptr() + 2), dict(texcoord_idx=d["tidx"].data_ptr() + 1),
                dict(texture=d["texture"].data_ptr() + 2), dict(texture=host_tex.ctypes.data),
                dict(texcoords=host_pts.ctypes.data),
                dict(point_idx=device_bad["point"].data_ptr()), dict(point_idx=device_bad["point_neg"].data_ptr()),
                dict(normal_idx=device_bad["normal"].data_ptr()), dict(texcoord_idx=device_bad["texcoord"].data_ptr()),
                dict(texcoord_idx=device_bad["texcoord_neg"].data_ptr()), dict(texture=device_bad["slot"].data_ptr()),
                dict(texture=device_bad["slot_empty"].data_ptr()),
                dict(points=db["points"].data_ptr(), num_points=len(big["points"]), point_idx=db["pidx"].data_ptr(),
                     num_tris=len(big["pidx"]), normals=None, normal_idx=None, texcoords=db["texcoords"].data_ptr(),
                     num_texcoords=len(big["texcoords"]), texcoord_idx=device_bad["grow"].data_ptr(), texture=None),
            ]
            for kw in cases:
                assert call(**kw) == A.RT_ERR_INVALID, kw
                assert mesh_bytes(ctx, 0) == before, kw
            replace(ctx, 0, g)
            check_arrays(ctx, ReplaceExpected(rt, sc, 0, g))
            # a good refit and update follow
            pts = deform(g["points"], "wobble")
            assert ctx.refit_mesh(0, to_dev(pts), d["pidx"]).item() == 0
            ctx.update_mesh(0, d["points"], d["pidx"])
            gu = dict(g); gu.pop("normals"); gu.pop("nidx")
            check_arrays(ctx, ReplaceExpected(rt, sc, 0, gu))
        # a mesh that two shapes reference, and a shape that is not a mesh
        dd = sc.desc.contents
        shapes = (A.rt_shape * (dd.num_shapes + 1))()
        C.memmove(shapes, dd.shapes, C.sizeof(A.rt_shape) * dd.num_shapes)
        shapes[dd.num_shapes] = shapes[0]
        desc2 = A.rt_scene_desc()
        C.memmove(C.byref(desc2), C.byref(dd), C.sizeof(desc2))
        desc2.shapes, desc2.num_shapes = shapes, dd.num_shapes + 1
        ctx2 = rt.GpuContext(0)
        try:
            ctx2.upload_scene(C.pointer(desc2))
            before2 = mesh_bytes(ctx2, 0)
            u = A.rt_mesh_update(d["points"].data_ptr(), P, d["pidx"].data_ptr(), T, None, 0, None)
            r = A.rt_mesh_replace(u, None, 0, None, None)
            assert ctx2._lib.rt_gpu_replace_mesh(ctx2.handle, 0, C.byref(r), None) == A.RT_ERR_INVALID
            assert mesh_bytes(ctx2, 0) == before2
        finally:
            ctx2.close()
        sph = make_scene(rt, [("sphere", (0.0, 0.0, 0.0), 1.0, ("diffuse", (1, 1, 1)))] + scenes.c1_torusknot(data_dir))
        ctx3 = rt.GpuContext(0)
        try:
            ctx3.upload_scene(sph)
            u = A.rt_mesh_update(d["points"].data_ptr(), P, d["pidx"].data_ptr(), T, None, 0, None)
            r = A.rt_mesh_replace(u, None, 0, None, None)
            assert ctx3._lib.rt_gpu_replace_mesh(ctx3.handle, 0, C.byref(r), None) == A.RT_ERR_INVALID
        finally:
            ctx3.close()
        # the torch layer
        before = mesh_bytes(ctx, 0)
        for kw in (dict(points=d["points"].cpu()), dict(point_idx=d["pidx"].long()), dict(texcoords=d["texcoords"], texcoord_idx=None),
                   dict(texcoords=None, texcoord_idx=d["tidx"]), dict(texcoords=d["points"]), dict(texcoord_idx=d["tidx"][:-1]),
                   dict(texture=d["texture"][:-1]), dict(texture=d["texture"].long()), dict(texture=d["texture"].cpu())):
            args = dict(points=d["points"], point_idx=d["pidx"], texcoords=d["texcoords"], texcoord_idx=d["tidx"],
                        texture=d["texture"])
            args.update(kw)
            with pytest.raises(ValueError):
                ctx.replace_mesh(0, **args)
        with pytest.raises(rt.RtError):
            ctx.replace_mesh(0, d["points"], d["pidx"], texture=device_bad["slot"])
        assert mesh_bytes(ctx, 0) == before
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 6. memory
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_replace_memory(rt, data_dir):
    """Scene bytes grow on a grow past the spare set's capacity, not on a shrink; twenty replaces alternating
    between two levels of detail stop growing them after the first two."""
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    small, mid, big = torus_sizes(sc)
    up = uploaded_geometry(sc, 0)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        b0 = scene_bytes(ctx)
        replace(ctx, 0, dict(up, points=deform(up["points"], "rigid")))      # the first replace allocates the spare set
        b1 = scene_bytes(ctx)
        assert b1 > b0
        replace(ctx, 0, geometry(grid(small)))            # shrink into the uploaded set
        assert scene_bytes(ctx) == b1
        replace(ctx, 0, geometry(grid(big)))              # grow past the spare set's capacity
        b2 = scene_bytes(ctx)
        assert b2 > b1
        replace(ctx, 0, geometry(grid(small, seed=1)))    # shrink
        replace(ctx, 0, geometry(grid(mid)))              # within capacity
        assert scene_bytes(ctx) == b2
        check_arrays(ctx, ReplaceExpected(rt, sc, 0, geometry(grid(mid))))
    finally:
        ctx.close()
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        lods = [geometry(grid(big), texcoords=True), geometry(grid(mid, seed=1), normals=True)]
        seen = []
        for k in range(20):
            replace(ctx, 0, lods[k % 2])
            seen.append(scene_bytes(ctx))
        assert seen[0] < seen[1], seen                    # the second level is larger than the uploaded set
        assert all(b == seen[1] for b in seen[1:]), seen
        check_arrays(ctx, ReplaceExpected(rt, sc, 0, lods[1]))
    finally:
        ctx.close()
