"""Appearance updates on the device (rt_gpu_update_materials / rt_gpu_update_lights / rt_gpu_update_texture and the
GpuContext wrappers).

The bar: after any sequence of updates every render, query and radiance call returns, bit for bit, what a fresh upload
of the edited description returns.  The expected side is a second context holding that fresh upload; the records and
texels the device holds are compared byte for byte through the debug hooks."""
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
PATH, PREVIEW, WHITTED, PRIMARY = 0, 1, 2, 3
DIFFUSE, CHECKER, REFLECTIVE, EMISSIVE, BLEND, COMBINE, NULL = range(7)


# ---------------------------------------------------------------------------------------------------
# no GPU: the struct layout and the texel table
# ---------------------------------------------------------------------------------------------------
def test_texture_update_layout_matches_c(rt):
    fields = ("x", "y", "width", "height", "rgba", "pitch", "texels8", "channels", "lut")
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rt_gpu.h"\nint main(void) {\n'
    src += '  printf("size %zu\\n", sizeof(rt_texture_update));\n'
    for f in fields:
        src += f'  printf("{f} %zu\\n", offsetof(rt_texture_update, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "u.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "u")
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        out = {k: int(v) for k, v in (line.split() for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())}
    u = rt._abi.rt_texture_update
    assert C.sizeof(u) == out["size"]
    for f in fields:
        assert getattr(u, f).offset == out[f], f


def test_texel_lut_is_the_loaders_table(rt, data_dir):
    lut = rt.texel_lut()
    assert lut.dtype == np.float32 and lut.shape == (512,)
    sc = rt.Scene(scenes.c3_unitychan(data_dir))
    m = sc.desc.contents.meshes[0]
    seen = 0
    for k in range(m.num_textures):
        t = m.textures[k]
        if bool(t.lut):
            assert np.ctypeslib.as_array(t.lut, (512,)).tobytes() == lut.tobytes()
            seen += 1
    assert seen > 0


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
def make_scene(rt, spec, unit_vectors=True):
    sc = rt.Scene(spec)
    if unit_vectors:
        sc.set_unit_vectors(seed=0, count=1 << 18)
    return sc


def copies(T, ptr, n):
    return [T.from_buffer_copy(ptr[i]) for i in range(n)]


class Edited:
    """A copy of a scene description (rt_scene_desc) whose materials, lights, shape records and texture slots can be
    edited: the fresh-upload side.  `keep` holds whatever owns the memory the description points into."""

    def __init__(self, rt, desc, keep=()):
        A = self.A = rt._abi
        d = self.d = desc
        self.keep = list(keep)
        self.materials = copies(A.rt_material, d.materials, d.num_materials)
        self.lights = copies(A.rt_light, d.lights, d.num_lights)
        self.shapes = copies(A.rt_shape, d.shapes, d.num_shapes)
        self.textures = [copies(A.rt_texture, d.meshes[i].textures, d.meshes[i].num_textures) for i in range(d.num_meshes)]

    def set_texels(self, mesh, slot, rgba):
        arr = np.ascontiguousarray(rgba, np.float32).copy()
        self.keep.append(arr)
        t = self.textures[mesh][slot]
        t.rgba = arr.ctypes.data_as(C.POINTER(C.c_float))
        t.texels8, t.lut, t.channels = None, None, 0

    def desc(self):
        A, d = self.A, self.d
        arr = lambda T, items: (T * max(len(items), 1))(*items)
        mats, lights, shapes = arr(A.rt_material, self.materials), arr(A.rt_light, self.lights), arr(A.rt_shape, self.shapes)
        meshes = (A.rt_mesh * max(d.num_meshes, 1))()
        C.memmove(meshes, d.meshes, C.sizeof(A.rt_mesh) * d.num_meshes)
        texs = []
        for i in range(d.num_meshes):
            texs.append(arr(A.rt_texture, self.textures[i]))
            meshes[i].textures = texs[-1]
            meshes[i].num_textures = len(self.textures[i])
        out = A.rt_scene_desc()
        C.memmove(C.byref(out), C.byref(d), C.sizeof(out))
        out.materials, out.num_materials = mats, len(self.materials)
        out.lights, out.num_lights = lights, len(self.lights)
        out.shapes, out.num_shapes = shapes, len(self.shapes)
        out.meshes = meshes
        self._hold = (mats, lights, shapes, meshes, texs)
        return out

    def fresh(self, rt):
        ctx = rt.GpuContext(0)
        ctx.upload_scene(C.pointer(self.desc()))
        return ctx


def frame(rt, ctx, mode, traverse=1, antialias=0, w=W, h=H, max_bounce=4):
    ctx.reset_accum(w, h)
    ctx.render_tile(rt.make_params(w, h, mode=mode, max_bounce=max_bounce, pass_count=1, antialias=antialias, seed=3,
                                   traverse=traverse))
    if mode == PRIMARY:
        return ctx.readback(rt.RT_READ_PRIMARY_IDS_I32X2, w, h), ctx.readback(rt.RT_READ_PRIMARY_DIST_F32, w, h)
    return ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, w, h)


def same_frames(a, b):
    if isinstance(a, tuple):
        return np.array_equal(a[0], b[0]) and same_bits(a[1], b[1])
    return same_bits(a, b)


RAYS = None


def rays_dev():
    global RAYS
    if RAYS is None:
        RAYS = to_dev(np.concatenate([pinhole_rays(W, H, True), random_rays(2048, 11)]))
    return RAYS


def check_all(rt, got, want, modes=(PATH, PREVIEW, WHITTED, PRIMARY), radiance=(PATH, PREVIEW, WHITTED)):
    """Renders in `modes` (both traversals, antialias 0 and 1), nearest-hit queries with hit11, occlusion queries and
    radiance in `radiance`, all bit for bit; the counters of the exact traversal's work equal."""
    import torch
    rays = rays_dev()
    for traverse in (0, 1):
        counters = []
        for ctx in (got, want):
            ctx.synchronize()
            ctx.reset_counters()
        for mode in modes:
            for aa in (0, 1):
                assert same_frames(frame(rt, got, mode, traverse, aa), frame(rt, want, mode, traverse, aa)), (mode, traverse, aa)
        res = []
        for ctx in (got, want):
            near = ctx.query_rays(rays, traverse=traverse)
            occ = ctx.query_rays(rays, any_hit=True, traverse=traverse)
            rad = [ctx.radiance_rays(rays, mode=m, max_bounce=4, seed=5, traverse=traverse) for m in radiance]
            torch.cuda.synchronize()
            ctx.synchronize()
            res.append((near["shape"].cpu().numpy(), near["tri"].cpu().numpy(), near["hit"].cpu().numpy(), occ.cpu().numpy(),
                        [r.cpu().numpy() for r in rad]))
            counters.append(ctx.counters())
        a, b = res
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1], b[1])
        assert same_bits(a[2], b[2])
        np.testing.assert_array_equal(a[3], b[3])
        for m, ra, rb in zip(radiance, a[4], b[4]):
            assert same_bits(ra, rb), (m, traverse)
        if traverse == 0:
            assert counters[0] == counters[1]


def check_records(ctx, ed):
    mats, lights = ctx.read_appearance()
    assert bytes(mats) == b"".join(bytes(m) for m in ed.materials)
    assert bytes(lights) == b"".join(bytes(l) for l in ed.lights)
    assert len(mats) == len(ed.materials) and len(lights) == len(ed.lights)


# material edits on a list of rt_material copies (in place); each keeps the graph valid
def _leaves(ms):
    return [i for i, m in enumerate(ms) if m.type not in (BLEND, COMBINE)]


def edit_colours(ms):
    for m in ms:
        m.rgb[0], m.rgb[1], m.rgb[2] = m.rgb[0] * 0.5, m.rgb[1] * 0.8, min(m.rgb[2] * 1.1 + 0.05, 1.0)


def edit_fuzz(ms):
    for m in ms:
        if m.type == REFLECTIVE:
            m.scalar = 0.35


def edit_checker(ms):
    for m in ms:
        if m.type == CHECKER:
            m.scalar = m.scalar * 2.5 + 0.5


def edit_blend(ms):
    for m in ms:
        if m.type == BLEND:
            m.scalar = 0.25


def edit_types(ms):
    """Diffuse -> Reflective, Reflective -> Null, Null -> Diffuse (first of each)."""
    firsts = {t: next((i for i, m in enumerate(ms) if m.type == t), None) for t in (DIFFUSE, REFLECTIVE, NULL)}
    for t, new in ((DIFFUSE, REFLECTIVE), (REFLECTIVE, NULL), (NULL, DIFFUSE)):
        i = firsts[t]
        if i is not None:
            ms[i].type, ms[i].scalar = new, 0.1


def edit_children(ms):
    leaves = _leaves(ms)
    for m in ms:
        if m.type == BLEND:
            m.child_a, m.child_b = m.child_b, m.child_a
        elif m.type == COMBINE:
            m.child_b = leaves[-1]


EDITS = {"colours": edit_colours, "fuzz": edit_fuzz, "checker": edit_checker, "blend": edit_blend, "types": edit_types,
         "children": edit_children}


def push_changes(ctx, before, after):
    """update_materials over the smallest range that holds every changed record."""
    changed = [i for i, (a, b) in enumerate(zip(before, after)) if bytes(a) != bytes(b)]
    if changed:
        lo, hi = changed[0], changed[-1]
        ctx.update_materials(after[lo:hi + 1], first=lo)


MAT_SCENES = {"default": scenes.default_scene, "mix": scenes.deterministic_mix, "unitychan": scenes.c3_unitychan}


# ---------------------------------------------------------------------------------------------------
# 1. material edits in place
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MAT_SCENES))
def test_material_edits_equal_fresh_upload(rt, data_dir, name):
    sc = make_scene(rt, MAT_SCENES[name](data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        check_records(ctx, ed)
        for edit, fn in EDITS.items():
            before = [type(m).from_buffer_copy(m) for m in ed.materials]
            fn(ed.materials)
            push_changes(ctx, before, ed.materials)
            check_records(ctx, ed)
            ref = ed.fresh(rt)
            try:
                check_all(rt, ctx, ref)
            finally:
                ref.close()
        # the Scene form: a host scene's flattened records
        ctx.update_materials(sc)
        ref = rt.GpuContext(0)
        try:
            ref.upload_scene(sc)
            check_records(ctx, Edited(rt, sc.desc.contents, (sc,)))
            check_all(rt, ctx, ref, modes=(PATH, WHITTED))
        finally:
            ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 2. appended nodes
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_appended_materials_and_shapes_pointing_at_them(rt, data_dir):
    A = rt._abi
    sc = make_scene(rt, scenes.default_scene(data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    n = len(ed.materials)
    new = [A.rt_material(REFLECTIVE, -1, -1, (0.9, 0.3, 0.2), 0.05), A.rt_material(DIFFUSE, -1, -1, (0.2, 0.4, 0.9), 0.0),
           A.rt_material(BLEND, n, n + 1, (0.0, 0.0, 0.0), 0.3), A.rt_material(COMBINE, n + 2, n, (0.0, 0.0, 0.0), 0.0)]
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        # refused before the append, accepted after
        rec = (A.rt_shape * 1)(ed.shapes[0])
        rec[0].material = n + 2
        assert ctx._lib.rt_gpu_update_shapes(ctx.handle, rec, 0, 1, None) == A.RT_ERR_INVALID
        ctx.update_materials(new[:2], first=n)                       # two appends, then two more past them
        ctx.update_materials(new[2:], first=n + 2)
        ed.materials += new
        check_records(ctx, ed)
        for k, mat in ((0, n + 2), (1, n + 3), (4, n)):
            ed.shapes[k].material = mat
            rec = (A.rt_shape * 1)(ed.shapes[k])
            ctx._check(ctx._lib.rt_gpu_update_shapes(ctx.handle, rec, k, 1, None))
        ref = ed.fresh(rt)
        try:
            check_all(rt, ctx, ref)
        finally:
            ref.close()
        rec = (A.rt_shape * 1)(ed.shapes[0])
        rec[0].material = n + 4
        assert ctx._lib.rt_gpu_update_shapes(ctx.handle, rec, 0, 1, None) == A.RT_ERR_INVALID
        # an edit that spans old and appended nodes
        span = [type(m).from_buffer_copy(m) for m in ed.materials[n - 2:]] + [A.rt_material(EMISSIVE, -1, -1, (0.5, 0.5, 0.1), 0.0)]
        span[0].rgb[0] = 0.123
        ctx.update_materials(span, first=n - 2)
        ed.materials[n - 2:] = span
        check_records(ctx, ed)
        ref = ed.fresh(rt)
        try:
            check_all(rt, ctx, ref, modes=(PATH, PREVIEW))
        finally:
            ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 3. rejected updates leave the scene exactly as it was
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rejected_material_updates_leave_the_scene(rt, data_dir):
    A = rt._abi
    lib = rt.load_library()
    sc = make_scene(rt, scenes.deterministic_mix(data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    ms = ed.materials
    n = len(ms)
    leaf = _leaves(ms)[0]
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        # eight nested Combines appended: a valid graph at the limit; the deepest one's child `leaf` is untouched
        chain = [A.rt_material(COMBINE, n + k + 1, leaf, (0, 0, 0), 0.0) for k in range(7)]
        chain.append(A.rt_material(COMBINE, leaf, leaf, (0, 0, 0), 0.0))
        ctx.update_materials(chain, first=n)
        ms += chain
        combine = next(i for i, m in enumerate(ms[:n]) if m.type == COMBINE)
        want_frames = {m: frame(rt, ctx, m) for m in (PATH, WHITTED)}

        def unchanged():
            check_records(ctx, ed)
            for m, f in want_frames.items():
                assert same_frames(frame(rt, ctx, m), f), m

        def bad(recs, first, count=None, what=""):
            arr = (A.rt_material * max(len(recs), 1))(*recs)
            rc = lib.rt_gpu_update_materials(ctx.handle, arr, first, len(recs) if count is None else count, None)
            assert rc == A.RT_ERR_INVALID, what
            assert lib.rt_gpu_last_error(ctx.handle), what
            unchanged()

        unchanged()
        # a cycle closed through a node the update does not touch: leaf -> combine -> (its child) ... -> leaf
        c = ms[combine]
        cyc = A.rt_material(BLEND, combine, combine, (0, 0, 0), 0.5)
        target = c.child_a if ms[c.child_a].type not in (BLEND, COMBINE) else c.child_b
        bad([cyc], target, what="cycle")
        assert b"cycle" in lib.rt_gpu_last_error(ctx.handle)
        # a ninth Combine reached through the update: the chain's shared leaf becomes a Combine
        other = _leaves(ms)[1]
        bad([A.rt_material(COMBINE, other, other, (0, 0, 0), 0.0)], leaf, what="nine combines")
        assert b"nests Combine" in lib.rt_gpu_last_error(ctx.handle)
        grown = len(ms)
        bad([A.rt_material(BLEND, 0, grown, (0, 0, 0), 0.5)], 0, what="child out of range")
        bad([A.rt_material(BLEND, 0, grown + 1, (0, 0, 0), 0.5)], grown, what="child out of range past the append")
        bad([A.rt_material(7, -1, -1, (1, 1, 1), 0.0)], 0, what="unknown type")
        bad([A.rt_material(-1, -1, -1, (1, 1, 1), 0.0)], 0, what="negative type")
        bad([A.rt_material(DIFFUSE, -1, -1, (1, 1, 1), 0.0)], grown + 1, what="first past the count")
        bad([A.rt_material(DIFFUSE, -1, -1, (1, 1, 1), 0.0)], -1, what="negative first")
        bad([A.rt_material(DIFFUSE, -1, -1, (1, 1, 1), 0.0)], 0, count=-1, what="negative count")
        assert lib.rt_gpu_update_materials(ctx.handle, None, 0, 1, None) == A.RT_ERR_INVALID
        unchanged()
        # still usable
        ms[0].rgb[1] = 0.01
        ctx.update_materials(ms[:1])
        ref = ed.fresh(rt)
        try:
            check_records(ctx, ed)
            check_all(rt, ctx, ref, modes=(PATH, WHITTED), radiance=(PATH,))
        finally:
            ref.close()
    finally:
        ctx.close()
    fresh_ctx = rt.GpuContext(0)
    try:
        m = (A.rt_material * 1)(A.rt_material(DIFFUSE, -1, -1, (1, 1, 1), 0.0))
        assert lib.rt_gpu_update_materials(fresh_ctx.handle, m, 0, 1, None) == A.RT_ERR_NO_SCENE
        assert lib.rt_gpu_update_lights(fresh_ctx.handle, None, 0, None) == A.RT_ERR_NO_SCENE
        u = A.rt_texture_update()
        assert lib.rt_gpu_update_texture(fresh_ctx.handle, 0, 0, C.byref(u), None) == A.RT_ERR_NO_SCENE
    finally:
        fresh_ctx.close()


# ---------------------------------------------------------------------------------------------------
# 4. the unit-vector table
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_diffuse_node_without_unit_vectors(rt, data_dir):
    A = rt._abi
    import torch
    sc = make_scene(rt, scenes.deterministic_mix(data_dir), unit_vectors=False)
    ed = Edited(rt, sc.desc.contents, (sc,))
    refl = next(i for i, m in enumerate(ed.materials) if m.type == REFLECTIVE)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        before = frame(rt, ctx, PATH)
        orig = A.rt_material.from_buffer_copy(ed.materials[refl])
        ed.materials[refl].type = DIFFUSE
        ctx.update_materials(ed.materials[refl:refl + 1], first=refl)       # accepted, as such an upload is
        with pytest.raises(rt.RtError):
            frame(rt, ctx, PATH)
        with pytest.raises(rt.RtError):
            ctx.radiance_rays(rays_dev(), mode=PATH)
        ref = ed.fresh(rt)
        try:
            with pytest.raises(rt.RtError):
                frame(rt, ref, PATH)
            check_all(rt, ctx, ref, modes=(PREVIEW, WHITTED, PRIMARY), radiance=(PREVIEW, WHITTED))
        finally:
            ref.close()
        ed.materials[refl] = orig
        ctx.update_materials([orig], first=refl)
        assert same_frames(frame(rt, ctx, PATH), before)
        torch.cuda.synchronize()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 5. lights
# ---------------------------------------------------------------------------------------------------
LIGHT_EDITS = [
    ("moved", [(0, (1.5, 4.0, 3.0), (1.0, 1.0, 1.0))]),
    ("recoloured", [(0, (1.5, 4.0, 3.0), (0.9, 0.3, 0.1))]),
    ("directional", [(1, (-0.3, -1.0, -0.5), (0.8, 0.8, 0.7))]),
    ("point_again", [(0, (-2.0, 3.0, 2.0), (0.6, 0.9, 0.6))]),
    ("five", [(0, (-2.0, 3.0, 2.0), (0.6, 0.9, 0.6)), (1, (0.2, -1.0, -0.3), (0.3, 0.3, 0.3)), (0, (3.0, 1.0, 4.0), (0.5, 0.2, 0.9)),
              (0, (0.0, 5.0, -2.0), (0.2, 0.2, 0.2)), (1, (1.0, -0.5, 0.0), (0.1, 0.4, 0.1))]),
    ("none", []),
    ("one_again", [(1, (0.0, -1.0, -1.0), (1.0, 1.0, 1.0))]),
]


def whitted_check(rt, got, want):
    import torch
    rays = rays_dev()
    for traverse in (0, 1):
        for ctx in (got, want):
            ctx.synchronize()
            ctx.reset_counters()
        for aa in (0, 1):
            assert same_frames(frame(rt, got, WHITTED, traverse, aa), frame(rt, want, WHITTED, traverse, aa)), (traverse, aa)
        rad = []
        for ctx in (got, want):
            r = ctx.radiance_rays(rays, mode=WHITTED, seed=5, traverse=traverse)
            torch.cuda.synchronize()
            ctx.synchronize()
            rad.append((r.cpu().numpy(), ctx.counters()))
        assert same_bits(rad[0][0], rad[1][0]), traverse
        assert rad[0][1]["shadow_rays"] == rad[1][1]["shadow_rays"] and rad[0][1]["rays"] == rad[1][1]["rays"]
        if traverse == 0:
            assert rad[0][1] == rad[1][1]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["torusknot", "mix"])
def test_light_edits_equal_upload_with_set_lights(rt, data_dir, name):
    spec = scenes.c1_torusknot(data_dir) if name == "torusknot" else scenes.deterministic_mix(data_dir)
    sc = make_scene(rt, spec)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for k, (what, lights) in enumerate(LIGHT_EDITS):
            sc2 = make_scene(rt, spec)
            sc2.set_lights(lights)
            # tuples and the Scene form in turn
            ctx.update_lights(lights if k % 2 == 0 else sc2)
            ed = Edited(rt, sc2.desc.contents, (sc2,))
            check_records(ctx, ed)
            assert len(ed.lights) == len(lights)
            ref = rt.GpuContext(0)
            try:
                ref.upload_scene(sc2)
                whitted_check(rt, ctx, ref)
            finally:
                ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 6. textures
# ---------------------------------------------------------------------------------------------------
def texture_slots(sc, mesh=0):
    d = sc.desc.contents
    m = d.meshes[mesh]
    return [k for k in range(m.num_textures) if bool(m.textures[k].rgba) or bool(m.textures[k].texels8)]


def kat_textures(rt, ctx, count):
    uv = np.stack(np.meshgrid(np.linspace(-0.25, 1.25, 41), np.linspace(-0.3, 1.3, 37)), -1).reshape(-1, 2).astype(np.float32)
    outs = []
    for k in range(count):
        out = np.zeros((len(uv), 4), np.float32)
        assert rt.load_library().rt_gpu_kat_texture(ctx.handle, k, uv.ctypes.data, len(uv), out.ctypes.data) == 0
        outs.append(out)
    return outs


@pytest.mark.gpu
def test_texture_updates_equal_fresh_upload(rt, data_dir):
    import torch
    A = rt._abi
    lib = rt.load_library()
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    lut = rt.texel_lut()
    rng = np.random.default_rng(7)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        slots = texture_slots(sc)
        assert len(slots) >= 4
        base = {k: ctx.read_texture(0, k) for k in slots}
        texels = {k: v.copy() for k, v in base.items()}
        s0, s1, s2, s3 = slots[:4]
        keep = []

        def keep_dev(a):
            keep.append(to_dev(a))
            return keep[-1]

        def put_float(slot, x, y, rgba):
            ctx.update_texture(0, slot, to_dev(rgba), x=x, y=y)
            texels[slot][y:y + rgba.shape[0], x:x + rgba.shape[1]] = rgba

        def put_bytes(slot, x, y, codes):
            ctx.update_texture(0, slot, to_dev(codes), x=x, y=y)
            c = codes.shape[2]
            codes = codes.astype(np.int64)
            v = np.stack([lut[codes[..., 0]], lut[codes[..., 1]], lut[codes[..., 2]],
                          lut[256 + codes[..., 3]] if c == 4 else np.ones(codes.shape[:2], np.float32)], -1)
            texels[slot][y:y + codes.shape[0], x:x + codes.shape[1]] = v

        # a full slot from floats
        h, w = texels[s0].shape[:2]
        put_float(s0, 0, 0, rng.random((h, w, 4), dtype=np.float32))
        # a rectangle whose rows are further apart than width * 16 bytes (the C call: the wrapper takes packed rows)
        h, w = texels[s1].shape[:2]
        rw, rh = w // 3, h // 4
        wide = torch.from_numpy(rng.random((rh, rw + 5, 4), dtype=np.float32)).to("cuda:0")
        u = A.rt_texture_update(3, 2, rw, rh, wide.data_ptr(), (rw + 5) * 16, None, 0, None)
        ctx._check(lib.rt_gpu_update_texture(ctx.handle, 0, s1, C.byref(u), ctx._torch_stream(torch.device("cuda", 0))))
        texels[s1][2:2 + rh, 3:3 + rw] = wide.cpu().numpy()[:, :rw]
        keep.append(wide)
        # 8-bit texels, 3 and 4 channels
        h, w = texels[s2].shape[:2]
        put_bytes(s2, 1, 1, rng.integers(0, 256, (h - 2, w - 3, 3), dtype=np.uint8))
        put_bytes(s2, w // 2, 0, rng.integers(0, 256, (h // 2, w // 2, 4), dtype=np.uint8))
        # rectangles on the right and bottom edges, and one texel
        h, w = texels[s3].shape[:2]
        put_float(s3, w - 7, 5, rng.random((9, 7, 4), dtype=np.float32))
        put_bytes(s3, 4, h - 6, rng.integers(0, 256, (6, 11, 4), dtype=np.uint8))
        put_float(s3, w - 1, h - 1, rng.random((1, 1, 4), dtype=np.float32))
        put_bytes(s3, 0, 0, rng.integers(0, 256, (1, 1, 3), dtype=np.uint8))
        # an empty rectangle is a no-op, in C and in the wrapper
        u = A.rt_texture_update(w, 0, 0, 4, keep_dev(rng.random((4, 1, 4), dtype=np.float32)).data_ptr(), 0, None, 0, None)
        ctx._check(lib.rt_gpu_update_texture(ctx.handle, 0, s3, C.byref(u), None))
        ctx.update_texture(0, s3, to_dev(np.zeros((0, 4, 4), np.float32)), x=w, y=0)

        for k in slots:
            got = ctx.read_texture(0, k)
            assert got.tobytes() == texels[k].tobytes(), k
            if k not in (s0, s1, s2, s3):
                assert got.tobytes() == base[k].tobytes(), k
            if k in (s0, s1, s2, s3):
                ed.set_texels(0, k, texels[k])
        ref = ed.fresh(rt)
        try:
            for k in slots:
                assert ref.read_texture(0, k).tobytes() == texels[k].tobytes(), k
            for a, b in zip(kat_textures(rt, ctx, len(slots)), kat_textures(rt, ref, len(slots))):
                assert same_bits(a, b)
            for mode in (PREVIEW, PATH):
                for aa in (0, 1):
                    assert same_frames(frame(rt, ctx, mode, 1, aa), frame(rt, ref, mode, 1, aa)), (mode, aa)
            check_all(rt, ctx, ref, modes=(PRIMARY,), radiance=(PREVIEW,))
        finally:
            ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 7. ordering across frame slots and streams, without host synchronisation
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_appearance_update_ordering_between_slots_and_streams(rt, data_dir):
    """Slot 0 renders a 1080p frame that is still running when each update returns (checked with an event); slot 1 and
    queries on the side stream, enqueued after the updates without a host synchronisation, see the new appearance."""
    import torch
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    edit_colours(ed.materials)
    edit_types(ed.materials)
    new_lights = [(0, (2.0, 3.0, 4.0), (0.9, 0.5, 0.2)), (1, (0.0, -1.0, -0.2), (0.3, 0.3, 0.5))]
    ed.lights = [rt.rt_light(k, v, c) for k, v, c in new_lights]
    slot = texture_slots(sc)[0]
    BW, BH = 1920, 1080
    big = rt.make_params(BW, BH, mode=PATH, max_bounce=6, pass_count=8, antialias=1, seed=3)
    small = rt.make_params(W, H, mode=WHITTED, max_bounce=6, pass_count=1, antialias=0, seed=3)

    def render(ctx, p):
        ctx.reset_accum(p.width, p.height)
        ctx.render_tile(p)
        return ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, p.width, p.height)

    old_ref = rt.GpuContext(0)
    ctx = rt.GpuContext(0)
    new_ref = None
    try:
        old_ref.upload_scene(sc)
        want_old = render(old_ref, big)
        ctx.upload_scene(sc)
        h, w = ctx.read_texture(0, slot).shape[:2]
        tex = np.random.default_rng(3).random((h, w, 4), dtype=np.float32)
        ed.set_texels(0, slot, tex)
        new_ref = ed.fresh(rt)
        want_new = render(new_ref, small)
        rays = rays_dev()
        want_q = new_ref.query_rays(rays)["hit"].cpu().numpy()
        want_r = new_ref.radiance_rays(rays, mode=PREVIEW, max_bounce=4, seed=5).cpu().numpy()
        for s, p in ((0, big), (1, small)):
            ctx.set_frame_slot(s)
            render(ctx, p)                                # warm-up: pools and buffers sized
            ctx.reset_accum(p.width, p.height)
            ctx.synchronize()
        d_tex = to_dev(tex)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        ctx.set_frame_slot(0)
        ctx.render_tile(big)                              # old appearance
        slot0 = torch.cuda.ExternalStream(ctx.stream)
        frame_done = torch.cuda.Event()
        frame_done.record(slot0)
        with torch.cuda.stream(side):
            ctx.update_materials(ed.materials)
            assert not frame_done.query(), "the slot-0 frame finished before the material update returned: make it larger"
            ctx.update_lights(new_lights)
            assert not frame_done.query(), "the slot-0 frame finished before the light update returned"
            ctx.update_texture(0, slot, d_tex)
            assert not frame_done.query(), "the slot-0 frame finished before the texture update returned"
            ctx.set_frame_slot(1)
            ctx.render_tile(small)                        # new appearance
            got_q = ctx.query_rays(rays)["hit"].cpu().numpy()
            got_r = ctx.radiance_rays(rays, mode=PREVIEW, max_bounce=4, seed=5).cpu().numpy()
        ctx.set_frame_slot(0)
        got_old = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, BW, BH)
        ctx.set_frame_slot(1)
        got_new = ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
        assert same_bits(got_old, want_old)
        assert same_bits(got_new, want_new)
        assert same_bits(got_q, want_q)
        assert same_bits(got_r, want_r)
    finally:
        ctx.close(); old_ref.close()
        if new_ref is not None:
            new_ref.close()


# ---------------------------------------------------------------------------------------------------
# 8. tiles
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_tiled_ranks_after_identical_updates(rt, data_dir):
    import torch
    sc = make_scene(rt, scenes.default_scene(data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    edit_colours(ed.materials)
    edit_children(ed.materials)
    lights = [(0, (1.0, 4.0, 2.0), (0.8, 0.7, 0.6)), (1, (0.5, -1.0, -0.5), (0.2, 0.2, 0.3))]
    slot = texture_slots(sc)[1]
    ranks = [rt.GpuContext(0) for _ in range(4)]
    TW, TH = 128, 96
    try:
        ranks[0].upload_scene(sc)
        h, w = ranks[0].read_texture(0, slot).shape[:2]
        codes = to_dev(np.random.default_rng(2).integers(0, 256, (h // 2, w // 2, 4), dtype=np.uint8))
        for ctx in ranks:
            ctx.upload_scene(sc)
            ctx.update_materials(ed.materials)
            ctx.update_lights(lights)
            ctx.update_texture(0, slot, codes, x=w // 4, y=h // 4)
        for mode in (PATH, WHITTED):
            kw = dict(mode=mode, max_bounce=5, antialias=1, pass_count=2, seed=6)
            ranks[0].reset_accum(TW, TH)
            ranks[0].render_tile(rt.make_params(TW, TH, **kw))
            full = ranks[0].readback(rt.RT_READ_ACCUM_RGBN_F32, TW, TH)
            dense = []
            for r, ctx in enumerate(ranks):
                p = rt.make_params(TW, TH, tile_size=16, tile_count=4, tile_rank=r, **kw)
                ctx.reset_accum(TW, TH)
                ctx.render_tile(p)
                buf = torch.empty((rt.owned_pixels(TW, TH, 16, 4, r), 4), dtype=torch.float32, device="cuda:0")
                ctx.pack_owned(p, buf.data_ptr(), buf.numel() * 4)
                ctx.synchronize()
                dense.append((p, buf))
            ranks[0].reset_accum(TW, TH)
            for r, (p, buf) in enumerate(dense):
                ranks[0].unpack_owned(p, r, buf.data_ptr(), buf.numel() * 4)
            ranks[0].synchronize()
            assert same_bits(ranks[0].readback(rt.RT_READ_ACCUM_RGBN_F32, TW, TH), full), mode
    finally:
        for ctx in ranks:
            ctx.close()


# ---------------------------------------------------------------------------------------------------
# 9. interleaved with mesh updates, refits and replaces; a re-upload starts clean
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mixed_sequence_with_mesh_updates(rt, data_dir):
    import torch
    from test_scene_updates import Expected, deform
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    d = sc.desc.contents
    shape = next(i for i in range(d.num_shapes) if d.shapes[i].type == rt._abi.RT_SHAPE_MESH)
    mesh = d.shapes[shape].mesh
    dump = sc.mesh_dump(shape)
    pts0, pidx = dump["points"], dump["pidx"].reshape(-1, 3)
    _, _, shade0 = sc.flat_mesh(mesh)
    dev = lambda a: to_dev(np.ascontiguousarray(a))
    lights = [(0, (-1.0, 3.0, 3.0), (0.7, 0.8, 0.9)), (0, (2.0, 1.0, 2.0), (0.4, 0.1, 0.1))]
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        slot = texture_slots(sc)[2]
        tex = ctx.read_texture(mesh, slot)
        mats = Edited(rt, d, (sc,)).materials
        edit_colours(mats)
        ctx.update_materials(mats)
        # the uploaded geometry again through a replace: its texture coordinates and slots from device memory
        ctx.replace_mesh(shape, dev(pts0), dev(pidx.astype(np.int32)), texcoords=dev(dump["texcoords"][:, :2]),
                         texcoord_idx=dev(dump["tidx"].reshape(-1, 3)), texture=dev(shade0["texture"].astype(np.int32)))
        codes = np.random.default_rng(4).integers(0, 256, (5, 9, 3), dtype=np.uint8)
        ctx.update_texture(mesh, slot, dev(codes), x=2, y=3)
        lut = rt.texel_lut()
        tex[3:8, 2:11] = np.stack([lut[codes[..., 0]], lut[codes[..., 1]], lut[codes[..., 2]], np.ones((5, 9), np.float32)], -1)
        status = ctx.refit_mesh(shape, dev(deform(pts0, "wobble")), dev(pidx.astype(np.int32)))
        ctx.update_lights(lights)
        final = deform(pts0, "rigid")
        ctx.update_mesh(shape, dev(final), dev(pidx.astype(np.int32)))
        edit_types(mats)
        ctx.update_materials(mats)
        torch.cuda.synchronize()
        assert int(status.cpu()[0]) == 0
        exp = Expected(rt, sc, shape, final)
        ed = Edited(rt, exp.desc, (exp,))
        ed.materials = mats
        ed.lights = [rt.rt_light(k, v, c) for k, v, c in lights]
        ed.set_texels(mesh, slot, tex)
        ref = ed.fresh(rt)
        try:
            check_records(ctx, ed)
            check_all(rt, ctx, ref, modes=(PATH, PREVIEW, WHITTED))
        finally:
            ref.close()
        # a re-upload starts clean
        ctx.upload_scene(sc)
        ref = rt.GpuContext(0)
        try:
            ref.upload_scene(sc)
            check_records(ctx, Edited(rt, d, (sc,)))
            for k in texture_slots(sc):
                assert ctx.read_texture(mesh, k).tobytes() == ref.read_texture(mesh, k).tobytes()
            check_all(rt, ctx, ref, modes=(PATH, WHITTED), radiance=(PATH, WHITTED))
        finally:
            ref.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------
# 10. errors of update_texture and of the wrappers
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_texture_update_errors(rt, data_dir):
    import torch
    A = rt._abi
    lib = rt.load_library()
    sc = make_scene(rt, scenes.c3_unitychan(data_dir))
    ed = Edited(rt, sc.desc.contents, (sc,))
    # one more slot, without pixels and named by no triangle: the upload accepts it, an update may not write it
    ed.textures[0].append(A.rt_texture())
    empty = len(ed.textures[0]) - 1
    ctx = ed.fresh(rt)
    try:
        slot = texture_slots(sc)[0]
        h, w = ctx.read_texture(0, slot).shape[:2]
        before = {k: ctx.read_texture(0, k) for k in texture_slots(sc)}
        good = torch.rand((2, 2, 4), device="cuda:0")
        codes = torch.randint(0, 256, (2, 2, 4), dtype=torch.uint8, device="cuda:0")
        lut = torch.from_numpy(rt.texel_lut()).to("cuda:0")
        host = np.zeros((4, 4, 4), np.float32)
        host_lut = rt.texel_lut()
        stream = ctx._torch_stream(torch.device("cuda", 0))

        def unchanged():
            for k, v in before.items():
                assert ctx.read_texture(0, k).tobytes() == v.tobytes(), k

        def call(mesh, s, u):
            return lib.rt_gpu_update_texture(ctx.handle, mesh, s, C.byref(u) if u is not None else None, stream)

        def rgba(x=0, y=0, wd=2, ht=2, ptr=None, pitch=32):
            return A.rt_texture_update(x, y, wd, ht, good.data_ptr() if ptr is None else ptr, pitch, None, 0, None)

        def bytes8(x=0, y=0, ch=4, lp=None, tp=None):
            return A.rt_texture_update(x, y, 2, 2, None, 0, codes.data_ptr() if tp is None else tp, ch,
                                       lut.data_ptr() if lp is None else lp)

        cases = [
            ("null update", 0, slot, None),
            ("mesh -1", -1, slot, rgba()), ("mesh past the end", 1, slot, rgba()),
            ("slot -1", 0, -1, rgba()), ("slot past the end", 0, empty + 1, rgba()), ("slot without pixels", 0, empty, rgba()),
            ("x < 0", 0, slot, rgba(x=-1)), ("y < 0", 0, slot, rgba(y=-1)), ("width < 0", 0, slot, rgba(wd=-1)),
            ("past the right edge", 0, slot, rgba(x=w - 1)), ("past the bottom edge", 0, slot, rgba(y=h - 1)),
            ("both sources", 0, slot, A.rt_texture_update(0, 0, 2, 2, good.data_ptr(), 32, codes.data_ptr(), 4, lut.data_ptr())),
            ("no source", 0, slot, A.rt_texture_update(0, 0, 2, 2, None, 32, None, 4, lut.data_ptr())),
            ("pitch below width * 16", 0, slot, rgba(pitch=31)), ("pitch not a multiple of 4", 0, slot, rgba(pitch=34)),
            ("misaligned rgba", 0, slot, rgba(ptr=good.data_ptr() + 2)),
            ("host rgba", 0, slot, rgba(ptr=host.ctypes.data, pitch=64)),
            ("2 channels", 0, slot, bytes8(ch=2)), ("5 channels", 0, slot, bytes8(ch=5)),
            ("no lut", 0, slot, A.rt_texture_update(0, 0, 2, 2, None, 0, codes.data_ptr(), 4, None)),
            ("misaligned lut", 0, slot, bytes8(lp=lut.data_ptr() + 2)),
            ("host lut", 0, slot, bytes8(lp=host_lut.ctypes.data)),
            ("host texels8", 0, slot, bytes8(tp=host.ctypes.data)),
            ("empty rectangle, host source", 0, slot, A.rt_texture_update(0, 0, 0, 0, host.ctypes.data, 0, None, 0, None)),
        ]
        for what, mesh, s, u in cases:
            assert call(mesh, s, u) == A.RT_ERR_INVALID, what
            assert lib.rt_gpu_last_error(ctx.handle), what
        unchanged()
        # the wrappers
        bad_tensors = [
            ("host tensor", torch.rand((2, 2, 4))),
            ("float64", torch.rand((2, 2, 4), dtype=torch.float64, device="cuda:0")),
            ("int32", torch.zeros((2, 2, 4), dtype=torch.int32, device="cuda:0")),
            ("float with 3 channels", torch.rand((2, 2, 3), device="cuda:0")),
            ("uint8 with 2 channels", torch.zeros((2, 2, 2), dtype=torch.uint8, device="cuda:0")),
            ("uint8 with 5 channels", torch.zeros((2, 2, 5), dtype=torch.uint8, device="cuda:0")),
            ("2-d", torch.zeros((2, 8), dtype=torch.uint8, device="cuda:0")),
            ("not contiguous", torch.rand((4, 2, 4), device="cuda:0")[::2]),
            ("numpy", np.zeros((2, 2, 4), np.float32)),
        ]
        for what, t in bad_tensors:
            with pytest.raises(ValueError):
                ctx.update_texture(0, slot, t)
        with pytest.raises(ValueError):
            ctx.update_texture(0, slot, codes, lut=lut[:256])
        with pytest.raises(ValueError):
            ctx.update_texture(0, slot, codes, lut=lut.cpu())
        with pytest.raises(rt.RtError):
            ctx.update_texture(0, slot, good, x=w - 1)
        with pytest.raises(rt.RtError):
            ctx.update_texture(0, empty, good)
        with pytest.raises(TypeError):
            ctx.update_materials([(0, -1, -1)])
        with pytest.raises(ValueError):
            ctx.update_materials(ed.materials[:1], count=2)
        with pytest.raises(ValueError):
            ctx.update_materials(sc, first=1, count=len(ed.materials))
        with pytest.raises(rt.RtError):
            ctx.update_materials(ed.materials[:1], first=len(ed.materials) + 1)
        with pytest.raises(ValueError):
            ctx.read_texture(0, empty)
        assert lib.rt_gpu_update_lights(ctx.handle, None, -1, None) == A.RT_ERR_INVALID
        assert lib.rt_gpu_update_lights(ctx.handle, None, 2, None) == A.RT_ERR_INVALID
        unchanged()
        check_records(ctx, ed)
        # still usable
        ctx.update_texture(0, slot, good, x=w - 2, y=h - 2)
        want = before[slot].copy()
        want[h - 2:, w - 2:] = good.cpu().numpy()
        assert ctx.read_texture(0, slot).tobytes() == want.tobytes()
    finally:
        ctx.close()
