"""Mesh refits on the device (rt_gpu_refit_mesh, GpuContext.refit_mesh).

The bar: a refit keeps the published tree's topology (node order, escapes, leaf order) and recomputes the triangle
records and node boxes from the new points.  refit_reference below states that in numpy; it is pinned to the host
builder on the uploaded points (no GPU).  On the device, the arrays equal the reference byte for byte, and every call
after a refit returns, bit for bit, what a fresh upload of the refit arrays returns."""
import ctypes as C

import numpy as np
import pytest

import scenes
from conftest import same_bits
from test_ray_queries import pinhole_rays, to_dev
from test_scene_updates import (SCENES, Expected, check_arrays, check_results, deform, fake_normals, fresh,
                                make_scene, mesh_shape)

F32 = np.float32
FLT_MAX = np.finfo(F32).max
FLT_EPSILON = np.finfo(F32).eps


# ---------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------
def refit_reference(nodes, tris, points, pidx):
    """The refit of a pre-order, escape-threaded tree (host layout: an inner node's `tri` is negative) to new points,
    in float32 with every multiply and add rounded on its own.  Returns (nodes, tris) with the topology's escape and
    tri words and leaf order."""
    pidx = np.asarray(pidx).reshape(-1, 3)
    points = np.asarray(points, F32)
    tris = tris.copy()
    t = tris["index"]
    p = [points[pidx[t, k]] for k in range(3)]
    tris["p0"], tris["p1"], tris["p2"] = p
    tris["pad0"] = tris["pad1"] = tris["pad2"] = 0
    a, b = p[1] - p[0], p[2] - p[0]
    n = np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1],
                  a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                  a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], 1)
    with np.errstate(all="ignore"):
        sqr = n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1] + n[:, 2] * n[:, 2]
        norm = ~(np.abs(sqr) < FLT_EPSILON)
        inv = F32(1.0) / np.sqrt(sqr)
        n[norm] = n[norm] * inv[norm, None]
    tris["n"] = n

    out = nodes.copy()
    N = len(nodes)
    bmin, bmax = np.empty((N, 3), F32), np.empty((N, 3), F32)
    tri = nodes["tri"]
    leaves = np.nonzero(tri >= 0)[0]
    slot = tri[leaves]
    mn, mx = np.full((len(leaves), 3), FLT_MAX, F32), np.full((len(leaves), 3), -FLT_MAX, F32)
    for k in range(3):                                   # RAabb's empty box expanded with p0, p1, p2 by < / >
        q = p[k][slot]
        mn = np.where(q < mn, q, mn)
        mx = np.where(q > mx, q, mx)
    bmin[leaves], bmax[leaves] = mn, mx
    # inner nodes, deepest first (children follow their parent in pre-order): left box, right only where strictly
    # smaller / larger
    inner = np.nonzero(tri < 0)[0]
    right = nodes["escape"][inner + 1]
    depth = [0] * N
    for i, r in zip(inner.tolist(), right.tolist()):
        depth[i + 1] = depth[r] = depth[i] + 1
    d_inner = np.array(depth)[inner]
    for d in range(int(d_inner.max(initial=0)), -1, -1):
        sel = d_inner == d
        i, L, R = inner[sel], inner[sel] + 1, right[sel]
        bmin[i] = np.where(bmin[R] < bmin[L], bmin[R], bmin[L])
        bmax[i] = np.where(bmax[R] > bmax[L], bmax[R], bmax[L])
    out["bmin"], out["bmax"] = bmin, bmax
    return out, tris


def refit_expected(rt, sc, shape, topo, points, pidx, normals=None, nidx=None):
    """Expected (the fresh-upload side) with the mesh's nodes and tris replaced by the refit of topology `topo`
    (host-layout nodes, tris)."""
    exp = Expected(rt, sc, shape, points, normals, nidx)
    exp.nodes, exp.tris = refit_reference(topo[0], topo[1], points, pidx)
    A = rt._abi
    m = exp.meshes[exp.mesh]
    m.nodes = exp.nodes.ctypes.data_as(C.POINTER(A.rt_bvh_node))
    m.tris = exp.tris.ctypes.data_as(C.POINTER(A.rt_tri))
    root = np.concatenate([exp.nodes[0]["bmin"], exp.nodes[0]["bmax"]]).astype(F32)
    exp.cull_scale = F32(max([F32(0.0)] + [abs(v) for v in root]))
    return exp


def refit(gpu, shape, points, pidx, normals=None, nidx=None):
    return gpu.refit_mesh(shape, to_dev(points), to_dev(np.asarray(pidx, np.int32).reshape(-1, 3)),
                          None if normals is None else to_dev(normals),
                          None if nidx is None else to_dev(np.asarray(nidx, np.int32).reshape(-1, 3)))


def host_topology(sc, shape):
    nodes, tris, _ = sc.flat_mesh(sc.desc.contents.shapes[shape].mesh)
    return nodes, tris


# ---------------------------------------------------------------------------------------------------
# 0. the reference against the host builder (no GPU)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["torusknot", "monkey_plane", "unitychan"])
def test_refit_reference_reproduces_host_build(rt, data_dir, name):
    """Refitting the uploaded tree to the uploaded points gives the host builder's triangle records byte for byte and
    its node boxes in value (the builder may pick the other sign of a zero bound)."""
    sc = rt.Scene(SCENES[name](data_dir))
    shape = mesh_shape(sc)
    dump = sc.mesh_dump(shape)
    nodes, tris = host_topology(sc, shape)
    got_nodes, got_tris = refit_reference(nodes, tris, dump["points"], dump["pidx"])
    assert got_tris.tobytes() == tris.tobytes()
    assert got_nodes["escape"].tobytes() == nodes["escape"].tobytes()
    assert got_nodes["tri"].tobytes() == nodes["tri"].tobytes()
    np.testing.assert_array_equal(got_nodes["bmin"], nodes["bmin"])
    np.testing.assert_array_equal(got_nodes["bmax"], nodes["bmax"])


# ---------------------------------------------------------------------------------------------------
# 1. arrays, 2. results
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_refit_arrays_equal_reference(rt, data_dir, name):
    sc = make_scene(rt, SCENES[name](data_dir))
    shape = mesh_shape(sc)
    dump = sc.mesh_dump(shape)
    pts0, pidx = dump["points"], dump["pidx"]
    topo = host_topology(sc, shape)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for kind in ("rigid", "wobble", "aniso", "degenerate"):
            pts = deform(pts0, kind)
            for with_normals in (False, True):
                nrm = fake_normals(pts, 1) if with_normals else None
                nidx = pidx.reshape(-1, 3) if with_normals else None
                status = refit(ctx, shape, pts, pidx, nrm, nidx)
                check_arrays(ctx, refit_expected(rt, sc, shape, topo, pts, pidx, nrm, nidx))
                assert status.item() == 0, (kind, with_normals)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_refit_results_equal_fresh_upload(rt, data_dir, name):
    sc = make_scene(rt, SCENES[name](data_dir))
    shape = mesh_shape(sc)
    dump = sc.mesh_dump(shape)
    pidx = dump["pidx"]
    topo = host_topology(sc, shape)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for kind, with_normals in (("wobble", False), ("rigid", True)):
            pts = deform(dump["points"], kind)
            nrm = fake_normals(pts, 2) if with_normals else None
            nidx = pidx.reshape(-1, 3) if with_normals else None
            refit(ctx, shape, pts, pidx, nrm, nidx)
            exp = refit_expected(rt, sc, shape, topo, pts, pidx, nrm, nidx)
            ref = fresh(rt, exp.desc)
            try:
                check_results(rt, ctx, ref)
            finally:
                ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 3. sequences with update_mesh in between
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refit_sequence(rt, data_dir):
    """upload -> refit -> refit -> update_mesh -> refit -> refit back to the uploaded points.  A refit keeps the
    topology it finds: the upload's, then the one update_mesh built (the host builder's for its points)."""
    sc = make_scene(rt, scenes.c1_torusknot(data_dir))
    dump = sc.mesh_dump(0)
    A, pidx = dump["points"], dump["pidx"]
    topo = host_topology(sc, 0)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for op, pts in (("refit", deform(A, "wobble")), ("refit", deform(A, "aniso")), ("update", deform(A, "rigid")),
                        ("refit", deform(A, "degenerate")), ("refit", A)):
            if op == "update":
                ctx.update_mesh(0, to_dev(pts), to_dev(pidx.reshape(-1, 3)))
                exp = Expected(rt, sc, 0, pts)
                topo = (exp.nodes, exp.tris)
            else:
                status = refit(ctx, 0, pts, pidx)
                exp = refit_expected(rt, sc, 0, topo, pts, pidx)
                assert status.item() == 0
            check_arrays(ctx, exp)
            ref = fresh(rt, exp.desc)
            try:
                check_results(rt, ctx, ref, modes=(0,))
            finally:
                ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 4. no host wait; ordering across frame slots and streams
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refit_returns_without_waiting(rt, data_dir):
    """With the torch stream held busy by a bounded sleep, refit_mesh returns while the stream is still busy (the
    first refit, which allocates the spare set, and a later one); once it drains the arrays are the refit's."""
    import torch
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    dump = sc.mesh_dump(0)
    pidx = dump["pidx"]
    topo = host_topology(sc, 0)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        d_idx = to_dev(pidx.reshape(-1, 3))
        for kind in ("wobble", "rigid"):
            pts = deform(dump["points"], kind)
            d_pts = to_dev(pts)
            torch.empty(1, dtype=torch.int32, device="cuda:0")          # the status block then comes from the cache
            torch.cuda.synchronize()
            stream = torch.cuda.current_stream(0)
            torch.cuda._sleep(200_000_000)                              # ~0.1 s at B200 clocks
            status = ctx.refit_mesh(0, d_pts, d_idx)
            busy = not stream.query()
            torch.cuda.synchronize()
            assert busy, f"{kind}: refit_mesh returned after its stream had drained"
            assert status.item() == 0
            check_arrays(ctx, refit_expected(rt, sc, 0, topo, pts, pidx))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_refit_ordering_between_slots_and_streams(rt, data_dir):
    """test_update_ordering_between_slots_and_streams with refit_mesh: a slot-0 frame still running when the refit
    returns sees the old geometry; slot 1 and a query on the side stream, enqueued after it, see the new one."""
    import torch
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    dump = sc.mesh_dump(0)
    pidx = dump["pidx"]
    new = deform(dump["points"], "rigid")
    exp = refit_expected(rt, sc, 0, host_topology(sc, 0), new, pidx)
    W, H = 64, 48
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
            status = ctx.refit_mesh(0, d_pts, d_idx)
            assert not frame_done.query(), "the slot-0 frame finished before the refit returned: make it larger"
            ctx.set_frame_slot(1)
            ctx.render_tile(small)                        # new geometry
            q = ctx.query_rays(rays)
            got_q = q["shape"].cpu().numpy()
            assert status.item() == 0
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
# 5. errors leave the mesh as it was
# ---------------------------------------------------------------------------------------------------
def mesh_bytes(ctx, mesh):
    return [np.asarray(a).tobytes() for a in ctx.read_mesh(mesh)]


@pytest.mark.gpu
def test_refit_host_rejections_leave_the_arrays(rt, data_dir):
    import torch
    A = rt._abi
    sc = make_scene(rt, scenes.deterministic_mix(data_dir))
    shape = mesh_shape(sc)
    mesh = sc.desc.contents.shapes[shape].mesh
    dump = sc.mesh_dump(shape)
    pts, pidx = deform(dump["points"], "wobble"), dump["pidx"].reshape(-1, 3).astype(np.int32)
    T = len(pidx)
    ctx = rt.GpuContext(0)
    try:
        status = torch.full((2,), 7, dtype=torch.int32, device="cuda:0")
        u = A.rt_mesh_update()
        assert ctx._lib.rt_gpu_refit_mesh(ctx.handle, shape, C.byref(u), status.data_ptr(), None) == A.RT_ERR_NO_SCENE
        ctx.upload_scene(sc)
        refit(ctx, shape, deform(dump["points"], "aniso"), pidx)          # a refit has happened: the spare set exists
        before = mesh_bytes(ctx, mesh)
        d_pts, d_idx = to_dev(pts), to_dev(pidx)
        d_nrm = to_dev(fake_normals(pts, 3))
        host_pts = np.ascontiguousarray(pts)
        host_status = np.zeros(2, np.int32)
        torch.cuda.synchronize()

        def call(shape=shape, points=d_pts.data_ptr(), num_points=len(pts), point_idx=d_idx.data_ptr(), num_tris=T,
                 normals=None, num_normals=0, normal_idx=None, status=status.data_ptr()):
            u = A.rt_mesh_update(points, num_points, point_idx, num_tris, normals, num_normals, normal_idx)
            return ctx._lib.rt_gpu_refit_mesh(ctx.handle, shape, C.byref(u), status, None)

        cases = [
            dict(points=None), dict(point_idx=None),
            dict(points=d_pts.data_ptr() + 2),                       # misaligned
            dict(points=host_pts.ctypes.data),                       # host memory
            dict(shape=0),                                           # a sphere
            dict(shape=-1), dict(shape=10_000),
            dict(num_tris=T - 1), dict(num_tris=T + 1), dict(num_points=0), dict(num_points=-3),
            dict(normals=d_nrm.data_ptr(), num_normals=len(pts)),    # normals without normal_idx
            dict(normal_idx=d_idx.data_ptr()),                       # and the reverse
            dict(status=status.data_ptr() + 2),                      # misaligned status
            dict(status=host_status.ctypes.data),                    # host status
        ]
        for kw in cases:
            assert call(**kw) == A.RT_ERR_INVALID, kw
            assert mesh_bytes(ctx, mesh) == before, kw
        assert status.cpu().tolist() == [7, 7]                   # nothing was enqueued
        assert ctx._lib.rt_gpu_refit_mesh(ctx.handle, shape, None, status.data_ptr(), None) == A.RT_ERR_INVALID
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
            before2 = mesh_bytes(ctx2, mesh)
            u = A.rt_mesh_update(d_pts.data_ptr(), len(pts), d_idx.data_ptr(), T, None, 0, None)
            assert ctx2._lib.rt_gpu_refit_mesh(ctx2.handle, shape, C.byref(u), None, None) == A.RT_ERR_INVALID
            assert mesh_bytes(ctx2, mesh) == before2
        finally:
            ctx2.close()
        # the torch layer
        for args in ((d_pts.cpu(), d_idx), (d_pts.double(), d_idx), (d_pts, d_idx.long()), (d_pts[:, :2], d_idx),
                     (d_pts, d_idx, d_nrm, None), (d_pts, d_idx, None, d_idx), (d_pts, d_idx.t()),
                     (d_pts, d_idx, d_nrm, d_idx[:-1]), (d_pts, d_idx, d_nrm.half(), d_idx),
                     (d_pts, d_idx.cpu())):
            with pytest.raises(ValueError):
                ctx.refit_mesh(shape, *args)
        with pytest.raises(rt.RtError):
            ctx.refit_mesh(0, d_pts, d_idx)                      # shape 0 is a sphere
        assert mesh_bytes(ctx, mesh) == before
    finally:
        ctx.close()


def with_nodes(rt, sc, nodes):
    """sc's description with mesh 0's node array replaced (the arrays must outlive the returned description)."""
    A = rt._abi
    d = sc.desc.contents
    meshes = (A.rt_mesh * d.num_meshes)()
    C.memmove(meshes, d.meshes, C.sizeof(meshes))
    meshes[0].nodes = nodes.ctypes.data_as(C.POINTER(A.rt_bvh_node))
    meshes[0].num_nodes = len(nodes)
    desc = A.rt_scene_desc()
    C.memmove(C.byref(desc), C.byref(d), C.sizeof(desc))
    desc.meshes = meshes
    return desc, meshes


@pytest.mark.gpu
def test_refit_rejects_trees_it_cannot_reach(rt, data_dir):
    """The upload accepts 2T-1-node trees in which a leaf slot is named twice or an inner node has an empty right range.
    A refit climbs from the leaf slots, so it would leave nodes of such a tree unwritten: it refuses them on the host,
    with the mesh untouched.  After update_mesh has built a tree, the refit works."""
    import torch
    A = rt._abi
    knot = rt.Scene(scenes.c1_torusknot(data_dir))
    nodes, _, _ = knot.flat_mesh(0)
    dup = nodes.copy()                                    # the leaf of slot 1 names slot 0 again
    dup["tri"][np.nonzero(dup["tri"] == 1)[0][0]] = 0
    pts2 = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.5]], np.float32)
    idx2 = np.array([[0, 1, 2], [1, 3, 2]], np.int32)
    two = rt.Scene()
    two.add_mesh_arrays(pts2, idx2, material=("diffuse", (1, 1, 1)))
    n2 = two.flat_mesh(0)[0]
    box = dict(bmin=n2[0]["bmin"], bmax=n2[0]["bmax"])
    same_slot = np.zeros(3, n2.dtype)                     # root, then two leaves of slot 0
    chain = np.zeros(3, n2.dtype)                         # root -> inner -> leaf: both right ranges empty
    for arr, esc, tri in ((same_slot, (3, 2, 3), (-1, 0, 0)), (chain, (3, 3, 3), (-1, -1, 0))):
        arr["escape"], arr["tri"] = esc, tri
        arr["bmin"], arr["bmax"] = box["bmin"], box["bmax"]
    for sc, arr in ((knot, dup), (two, same_slot), (two, chain)):
        dump = sc.mesh_dump(0)
        pidx = dump["pidx"].reshape(-1, 3).astype(np.int32)
        pts = deform(dump["points"], "wobble")
        d_pts, d_idx = to_dev(pts), to_dev(pidx)
        status = torch.full((1,), 7, dtype=torch.int32, device="cuda:0")
        desc, keep = with_nodes(rt, sc, arr)
        ctx = rt.GpuContext(0)
        try:
            ctx.upload_scene(C.pointer(desc))
            before = mesh_bytes(ctx, 0)
            torch.cuda.synchronize()
            u = A.rt_mesh_update(d_pts.data_ptr(), len(pts), d_idx.data_ptr(), len(pidx), None, 0, None)
            assert ctx._lib.rt_gpu_refit_mesh(ctx.handle, 0, C.byref(u), status.data_ptr(), None) == A.RT_ERR_INVALID
            with pytest.raises(rt.RtError):
                ctx.refit_mesh(0, d_pts, d_idx)
            assert mesh_bytes(ctx, 0) == before
            assert status.item() == 7                     # nothing was enqueued
            ctx.update_mesh(0, d_pts, d_idx)
            topo = Expected(rt, sc, 0, pts)
            again = deform(dump["points"], "aniso")
            assert refit(ctx, 0, again, pidx).item() == 0
            check_arrays(ctx, refit_expected(rt, sc, 0, (topo.nodes, topo.tris), again, pidx))
        finally:
            ctx.close()


@pytest.mark.gpu
def test_refit_bad_indices_leave_the_scene(rt, data_dir):
    """Indices out of range are found on the device: status 1 (point) or 2 (normal), the mesh and every result as they
    were.  After one and after two bad refits in a row, a good refit and an update_mesh still give the expected
    arrays: the spare / published bookkeeping stayed consistent."""
    sc = make_scene(rt, scenes.deterministic_mix(data_dir))
    shape = mesh_shape(sc)
    mesh = sc.desc.contents.shapes[shape].mesh
    dump = sc.mesh_dump(shape)
    pts0, pidx = dump["points"], dump["pidx"].reshape(-1, 3).astype(np.int32)
    T, P = len(pidx), len(pts0)
    bad_idx = pidx.copy(); bad_idx[T // 2, 1] = P
    neg_idx = pidx.copy(); neg_idx[T - 1, 2] = -1
    big_nidx = pidx.copy(); big_nidx[3, 0] = P + 1_000_000        # far outside normals: must never be loaded
    neg_nidx = pidx.copy(); neg_nidx[0, 0] = -(1 << 30)
    topo = host_topology(sc, shape)
    ctx, ref = rt.GpuContext(0), rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        ref.upload_scene(sc)

        def bad(want, pts, idx, nrm=None, nidx=None):
            before = mesh_bytes(ctx, mesh)
            status = refit(ctx, shape, pts, idx, nrm, nidx)
            assert status.item() == want
            assert mesh_bytes(ctx, mesh) == before

        def good(kind):
            nonlocal topo
            pts = deform(pts0, kind)
            status = refit(ctx, shape, pts, pidx)
            assert status.item() == 0
            exp = refit_expected(rt, sc, shape, topo, pts, pidx)
            check_arrays(ctx, exp)
            return exp

        def update(kind):
            nonlocal topo
            pts = deform(pts0, kind)
            ctx.update_mesh(shape, to_dev(pts), to_dev(pidx))
            exp = Expected(rt, sc, shape, pts)
            check_arrays(ctx, exp)
            topo = (exp.nodes, exp.tris)

        w = deform(pts0, "wobble")
        nrm = fake_normals(w, 4)
        # on the uploaded arrays, before any spare set exists
        bad(1, w, bad_idx)
        bad(1, w, neg_idx)
        bad(2, w, pidx, nrm, big_nidx)
        bad(2, w, pidx, nrm, neg_nidx)
        bad(3, w, bad_idx, nrm, big_nidx)
        check_results(rt, ctx, ref)
        # one bad refit, then a good refit and an update
        good("rigid")
        bad(1, w, bad_idx)
        good("aniso")
        update("wobble")
        # two bad refits in a row, then a good refit and an update
        bad(2, w, pidx, nrm, big_nidx)
        bad(1, w, neg_idx)
        exp = good("degenerate")
        update("rigid")
        exp = good("aniso")
        want = fresh(rt, exp.desc)
        try:
            check_results(rt, ctx, want, modes=(0,))
        finally:
            want.close()
    finally:
        ctx.close(); ref.close()
