"""The ray primitives, slab tests and texture sampler of rt_device.cuh at their numeric edges, and the refusal of
non-finite mesh geometry.

Random rays and primitives (tests/test_gpu_parity.py) almost never produce an exact zero, a tangent, an origin on a
face or a plane, a direction component at the FLT_EPSILON cut-off, an overflow, a NaN or an infinity; those are the
inputs where a GPU build and an x86 build can disagree.  Here seeded generators produce them on purpose and the device
functions (rt_gpu_kat, rt_gpu_kat_texture) are compared bit for bit with the `ref` fixture (NaNs in position only).

The walks rely on two invariants that the upload, the mesh edits and the device builder enforce by refusing NaN and
infinite coordinates: slab_fast equals the reference's slab test on finite boxes, and the culled walk's margin holds
for triangles with a finite face normal (the CULL paragraph of rt_device.cuh).  The mesh-level tests hold every walk
kernel to the restatement on accepted boundary meshes, and check each refusal.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import bits, same_bits

F = np.float32
FMAX = np.finfo(F).max
EPS = np.finfo(F).eps
TINY = np.finfo(F).tiny                 # smallest normal
DENORM = F(1e-40)
INF, NAN = F(np.inf), F(np.nan)


def up(x):
    return np.nextafter(F(x), F(np.inf))


def down(x):
    return np.nextafter(F(x), F(-np.inf))


class Cases:
    """Rows of rays (7 floats) and primitives, each tagged with the edge it exercises."""

    def __init__(self, width):
        self.width, self.rays, self.prims, self.tags = width, [], [], []

    def add(self, tag, o, d, dist, prim):
        self.rays.append([*o, *d, dist])
        self.prims.append(list(prim))
        self.tags.append(tag)

    def arrays(self):
        rays = np.array(self.rays, np.float64).astype(F)
        prims = np.array(self.prims, np.float64).astype(F).reshape(-1, self.width)
        return rays, prims, np.array(self.tags)


def octants():
    return [np.array([sx, sy, sz], F) for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)]


def slab_cases(seed=0):
    rng = np.random.default_rng(seed)
    c = Cases(6)
    rnd = lambda *s: rng.normal(size=s).astype(F)
    for _ in range(4):
        lo = rnd(3)
        hi = lo + np.abs(rnd(3)) + F(0.25)
        box = [*lo, *hi]
        for sgn in octants():
            d = sgn * (np.abs(rnd(3)) + F(0.05))
            for face in range(6):
                o = (lo + hi) * F(0.5) + rnd(3) * F(0.1)
                o[face % 3] = (lo if face < 3 else hi)[face % 3]
                c.add("face_origin", o, d, F(10), box)
                c.add("face_origin", o, -d, F(10), box)
        for k, tag in ((1, "flat1"), (2, "flat2"), (3, "flat3")):
            fl = hi.copy()
            fl[:k] = lo[:k]
            for _ in range(6):
                o = lo + rnd(3) * F(2)
                target = (lo + fl) * F(0.5)
                c.add(tag, o, target - o, F(10), [*lo, *fl])
            o = lo.copy()
            c.add(tag, o, rnd(3), F(10), [*lo, *fl])       # origin on the flat box
    for _ in range(8):
        o, d = rnd(3), rnd(3)
        c.add("empty", o, d, F(10), [FMAX, FMAX, FMAX, -FMAX, -FMAX, -FMAX])
        lo = rnd(3)
        c.add("inverted", o, d, F(10), [*(lo + F(1)), *lo])
        c.add("inverted", o, d, F(10), [lo[0], lo[1] + F(1), lo[2], lo[0] + F(1), lo[1], lo[2] + F(1)])
    for sgn in octants():
        d = sgn * (np.abs(rnd(3)) + F(0.01))
        for box in ([-FMAX, -FMAX, -FMAX, FMAX, FMAX, FMAX], [FMAX * F(0.5), -FMAX, -FMAX, FMAX, FMAX, FMAX],
                    [-FMAX, -FMAX, -FMAX, -FMAX * F(0.75), FMAX, F(1)]):
            for o in (rnd(3), np.array([-FMAX * F(0.9), FMAX * F(0.9), F(0)], F), np.array([FMAX, -FMAX, FMAX], F)):
                c.add("huge", o, d, FMAX, box)
    lo, hi = np.array([-1, -1, -1], F), np.array([1, 1, 1], F)
    for v in (EPS, down(EPS), up(EPS), -EPS, down(-EPS), up(-EPS)):
        for axis in range(3):
            d = rnd(3)
            d[axis] = v
            for o in (rnd(3) * F(0.5), rnd(3) * F(3), np.array([0, 0, -5], F)):
                c.add("eps_dir", o, d, F(100), [*lo, *hi])
                c.add("eps_dir", o, d, F(100), [*(lo + F(1.5)), *(hi + F(1.5))])
    for v in (F(0), F(-0.0), DENORM, -DENORM, TINY):
        for axis in range(3):
            d = rnd(3)
            d[axis] = v
            for o in (rnd(3) * F(0.5), rnd(3) * F(3)):
                c.add("zero_dir", o, d, F(10), [*lo, *hi])
    for bad in (NAN, INF, -INF):
        for k in range(6):
            o, d = rnd(3) * F(2), rnd(3)
            (o if k < 3 else d)[k % 3] = bad
            c.add("nonfinite_ray", o, d, F(10), [*lo, *hi])
    o, d = np.array([0, 0, -5], F), np.array([0.1, 0.1, 0.99], F)
    for bad in (NAN, INF, -INF):
        for k in range(6):
            box = [*lo, *hi]
            box[k] = bad
            c.add("nonfinite_box", o, d, F(10), box)           # the issue's ray: bmax.x = NaN enters under the reference
            c.add("nonfinite_box", rnd(3) * F(3), rnd(3), F(10), box)
    return c.arrays()


def triangle_cases(seed=1):
    rng = np.random.default_rng(seed)
    c = Cases(9)
    rnd = lambda *s: rng.normal(size=s).astype(F)
    for _ in range(6):
        p = rnd(3, 3)
        q = rnd(3, 3)
        q[0], q[1] = p[0], p[1]                             # two triangles sharing the edge p0-p1
        for tri in (p, q):
            for k in range(3):
                o = rnd(3) * F(4)
                c.add("vertex", o, tri[k] - o, F(3), tri.reshape(-1))
            mid = (p[0] + p[1]) * F(0.5)
            o = rnd(3) * F(4)
            c.add("shared_edge", o, mid - o, F(3), tri.reshape(-1))
            c.add("shared_edge", p[0] - (p[1] - p[0]), p[1] - p[0], F(3), tri.reshape(-1))   # along the edge
    flat = np.array([[-1, -1, 0], [1, -1, 0], [0, 1, 0]], F)
    for _ in range(6):
        x, y = rng.uniform(-0.5, 0.5, 2).astype(F)
        for tri in (flat, flat[::-1].copy()):
            c.add("end_on_plane", [x, y, 1], [0, 0, -1], F(1), tri.reshape(-1))
            c.add("end_on_plane", [x, y, 1], [0, 0, -0.5], F(2), tri.reshape(-1))
            c.add("origin_on_plane", [x, y, 0], [0, 0, -1], F(1), tri.reshape(-1))
            c.add("origin_on_plane", [x, y, F(-0.0)], [0, 0, 1], F(1), tri.reshape(-1))
            for D in (EPS, down(EPS), up(EPS), F(2) * EPS):
                c.add("d3_eps", [x, y, EPS / F(4)], [0, 0, -1], D, tri.reshape(-1))
                c.add("d3_eps", [x, y, EPS / F(4)], [0, 0, -4], D / F(4), tri.reshape(-1))
            for D in (F(0), F(-0.0), F(-1), F(-5), INF):
                c.add("dist_edge", [x, y, 1], [0, 0, -1], D, tri.reshape(-1))
                c.add("dist_edge", [x, y, -1], [0, 0, -1], D, tri.reshape(-1))
    for _ in range(6):
        a = rnd(3)
        b = a + rnd(3)
        o = rnd(3) * F(3)
        for tri in (np.stack([a, a, a]), np.stack([a, b, a + (b - a) * F(2)])):
            c.add("zero_area", o, a - o, F(5), tri.reshape(-1))
            c.add("zero_area", o, rnd(3), F(5), tri.reshape(-1))
        den = (rnd(3, 3) * DENORM).astype(F)
        c.add("denormal", [0, 0, 1], [0, 0, -1], F(2), den.reshape(-1))
        c.add("denormal", [DENORM, 0, 1], [0, 0, -1], F(2), (flat * DENORM).reshape(-1))
        c.add("denormal", [0, 0, 1], [DENORM, -DENORM, -1], F(2), flat.reshape(-1))
    for k in range(9):
        tri = flat.reshape(-1).copy()
        tri[k] = NAN
        for o, d in (([0.1, 0.1, 1], [0, 0, -1]), ([0.1, 0.1, -1], [0, 0, 1]), ([5, 5, 5], [1, 1, 1]), ([0, 0, 3], [0, 0, 1])):
            c.add("nan_corner", o, d, F(4), tri)
    return c.arrays()


def sphere_cases(seed=2):
    rng = np.random.default_rng(seed)
    c = Cases(4)
    for r in (1, 2, 3, 5):
        for k in (4, 10, 20):
            for rad in (F(r), down(F(r)), up(F(r))):
                c.add("tangent", [-k, r, 0], [1, 0, 0], F(1), [0, 0, 0, rad])
                c.add("tangent", [0, -k, r], [0, 1, 0], F(2 * k), [0, 0, 0, rad])
    for _ in range(8):
        d = rng.normal(size=3).astype(F)
        rad = F(abs(rng.normal()) + 0.5)
        c.add("origin_on_surface", [rad, 0, 0], d, F(10), [0, 0, 0, rad])
        c.add("origin_on_surface", [0, -rad, 0], d, F(10), [0, 0, 0, rad])
        c.add("origin_inside", rng.normal(size=3).astype(F) * rad * F(0.3), d, F(10), [0, 0, 0, rad])
        o = rng.normal(size=3).astype(F) * F(3)
        for rad in (F(0), F(-0.0), F(-1), F(-2.5)):
            c.add("radius_edge", o, -o, F(2), [0, 0, 0, rad])
    for D in (F(9), down(F(9)), up(F(9))):
        c.add("dist_equal", [-10, 0, 0], [1, 0, 0], D, [0, 0, 0, 1])
        c.add("dist_equal", [0, 0, -10], [0, 0, 1], D, [0, 0, 0, 1])
        c.add("dist_equal", [0, -7, 0], [0, 0.5, 0], D * F(2) / F(3), [0, 0, 0, 1])
    return c.arrays()


def plane_cases(seed=3):
    rng = np.random.default_rng(seed)
    c = Cases(6)
    e6 = F(1e-6)
    for v in (e6, down(e6), up(e6), down(down(e6)), up(up(e6)), -e6, down(-e6), up(-e6)):
        c.add("denom_1e6", [0, 1, 0], [1, v, 0], F(1e9), [0, 1, 0, 0, 0, 0])
        c.add("denom_1e6", [0, -1, 0], [1, v, 0], F(1e9), [0, 1, 0, 0, 0, 0])
    for _ in range(6):
        o = rng.normal(size=3).astype(F)
        o[1] = 0
        d = rng.normal(size=3).astype(F)
        c.add("t_zero", o, d, F(5), [0, 1, 0, 0, 0, 0])
        c.add("parallel_inside", o, [d[0], 0, d[2]], F(5), [0, 1, 0, 0, 0, 0])
        c.add("parallel_inside", o, [d[0], F(-0.0), d[2]], F(5), [0, 1, 0, 0, 0, 0])
    for D in (F(1), down(F(1)), up(F(1)), F(3), up(F(3))):
        c.add("t_dist", [0, 1, 0], [0, -1, 0], D, [0, 1, 0, 0, 0, 0])
        c.add("t_dist", [0.5, 3, 0.5], [0, -1, 0], D, [0, 1, 0, 0, 0, 0])
    return c.arrays()


def capsule_cases(seed=4):
    rng = np.random.default_rng(seed)
    c = Cases(7)
    for _ in range(6):
        a = rng.normal(size=3).astype(F)
        o = rng.normal(size=3).astype(F) * F(3)
        c.add("degenerate_axis", o, a - o, F(10), [*a, *a, F(0.5)])
        c.add("degenerate_axis", o, rng.normal(size=3).astype(F), F(10), [*a, *a, F(0.5)])
        for tilt in (F(0), EPS, F(2) * EPS, F(3e-4), F(4e-4), F(5e-4)):
            c.add("parallel_axis", [0.2, 0, -5], [tilt, 0, 1], F(20), [0, 0, 0, 0, 0, 1, F(0.5)])
            c.add("parallel_axis", [0.7, 0, -5], [0, tilt, 1], F(20), [0, 0, 0, 0, 0, 1, F(0.5)])
        c.add("origin_on_cylinder", [0.5, 0, 0.5], rng.normal(size=3).astype(F), F(10), [0, 0, 0, 0, 0, 1, F(0.5)])
        c.add("origin_on_cylinder", [0, -0.5, 0.25], [0, 1, 0], F(10), [0, 0, 0, 0, 0, 1, F(0.5)])
        c.add("radius_zero", o, -o, F(10), [0, 0, -1, 0, 0, 1, F(0)])
        c.add("radius_zero", [1, 0, 0], [-1, 0, 0], F(10), [0, 0, -1, 0, 0, 1, F(0)])
    return c.arrays()


def scalar_edges():
    v = [F(0), F(-0.0), DENORM, -DENORM, F(1e-45), TINY, INF, -INF, NAN, FMAX, -FMAX, F(1), F(-1)]
    v += [F(2.0) ** k for k in range(-149, 128, 7)]
    return np.array(v, F)


def barycentric_cases():
    rows, tags = [], []
    a, b, c = [0, 0, 0], [1, 0, 0], [0, 1, 0]
    for s in scalar_edges():
        rows.append([s, s, s, *a, *b, *c]); tags.append("scalar_point")
        rows.append([0.25, 0.25, 0, *a, s, 0, 0, *c]); tags.append("scalar_corner")
    for t in (F(0), F(2), F(-1), F(0.5)):
        rows.append([1, 1, 0, 0, 0, 0, 1, 1, 1, 2 * t, 2 * t, 2 * t]); tags.append("collinear")   # denominator 0
        rows.append([1, 1, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1]); tags.append("collinear")
    return np.array(rows, np.float64).astype(F), np.array(tags)


PRIMS = {"slab": (0, 6, slab_cases), "triangle": (1, 9, triangle_cases), "sphere": (2, 4, sphere_cases),
         "plane": (3, 6, plane_cases), "capsule": (4, 7, capsule_cases)}
REF_FN = {"slab": "kat_aabb", "triangle": "kat_triangle", "sphere": "kat_sphere", "plane": "kat_plane", "capsule": "kat_capsule"}
EXPECTED_TAGS = {
    "slab": {"face_origin", "flat1", "flat2", "flat3", "empty", "inverted", "huge", "eps_dir", "zero_dir", "nonfinite_ray",
             "nonfinite_box"},
    "triangle": {"vertex", "shared_edge", "end_on_plane", "origin_on_plane", "d3_eps", "dist_edge", "zero_area", "denormal",
                 "nan_corner"},
    "sphere": {"tangent", "origin_on_surface", "origin_inside", "radius_edge", "dist_equal"},
    "plane": {"denom_1e6", "t_zero", "t_dist", "parallel_inside"},
    "capsule": {"degenerate_axis", "parallel_axis", "origin_on_cylinder", "radius_zero"},
}


# ---- CPU: the generators reach every edge; the restatement equals the compiled reference on them ---------------------
def test_generators_reach_every_edge():
    for name, (_, width, gen) in PRIMS.items():
        rays, prims, tags = gen()
        assert rays.shape == (len(tags), 7) and prims.shape == (len(tags), width)
        assert set(tags) == EXPECTED_TAGS[name], name
    rays, prims, tags = slab_cases()
    d = rays[:, 3:6]
    assert np.any(d == EPS) and np.any(d == -EPS) and np.any(d == up(EPS)) and np.any(d == down(EPS))
    assert np.any((d == 0) & np.signbit(d)) and np.any(np.abs(d) == DENORM)
    assert np.isnan(prims).any() and np.isinf(prims).any() and np.isnan(rays).any()
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        t = (prims[:, :3] - rays[:, :3]) / d
    assert np.isinf(t[tags == "huge"]).any()                   # (b - o) * inv overflows
    o, b = rays[tags == "face_origin", :3], prims[tags == "face_origin"]
    assert np.all(np.any(o == b[:, :3], 1) | np.any(o == b[:, 3:], 1))
    rays, prims, tags = triangle_cases()
    assert np.isnan(prims[tags == "nan_corner"]).any(1).all()
    assert set(rays[tags == "dist_edge", 6].tolist()) >= {0.0, -1.0, np.inf}
    rays, prims, tags = sphere_cases()
    # integer geometry: the tangent discriminant b*b - 4*a*c is exactly 0 in fp32 on the unperturbed rows
    tan = (tags == "tangent") & (prims[:, 3] == np.round(prims[:, 3]))
    r, p = rays[tan], prims[tan]
    dxyz = r[:, 3:6] * r[:, 6:7]
    a = (dxyz * dxyz).sum(1, dtype=F)
    b = (F(2) * dxyz * (r[:, :3] - p[:, :3])).sum(1, dtype=F)
    cc = (r[:, :3] * r[:, :3]).sum(1, dtype=F) - p[:, 3] * p[:, 3]
    assert np.all(b * b - F(4) * a * cc == 0)
    x = scalar_edges()
    assert np.isnan(x).any() and np.isinf(x).any() and (x == FMAX).any() and np.any((x == 0) & np.signbit(x))
    assert "collinear" in set(barycentric_cases()[1])


def test_restatement_equals_reference_on_edges(port):
    from oracle import bindings
    if not bindings.ref_available():
        pytest.skip("oracle/_ref/libref_oracle.so not built")
    from conftest import _ref_oracle
    ref = _ref_oracle(False)
    for name, (_, _, gen) in PRIMS.items():
        rays, prims, _ = gen()
        f1, o1 = getattr(port, REF_FN[name])(rays, prims)
        f2, o2 = getattr(ref, REF_FN[name])(rays, prims)
        np.testing.assert_array_equal(f1, f2, err_msg=name)
        assert same_bits(o1, o2), name
    x = scalar_edges()
    assert same_bits(port.kat_qrsqrt(x), ref.kat_qrsqrt(x))
    pabc, _ = barycentric_cases()
    assert same_bits(port.kat_barycentric(pabc), ref.kat_barycentric(pabc))


def nan_mesh(bad=NAN):
    pts = np.array([[-1, -1, 0], [1, -1, 0], [0, 1, 0], [2, 2, 1], [3, 2, 1], [2, 3, 1]], F)
    pts[4, 1] = bad
    return pts, np.array([[0, 1, 2], [3, 4, 5]], np.int32)


def test_host_layer_builds_a_tree_for_a_nan_mesh(rt, tmp_path):
    """The loader and the host builder take non-finite points and terminate; the upload is what refuses them."""
    obj = tmp_path / "nan.obj"
    obj.write_text("v 0 0 0\nv 1 0 0\nv nan 1 0\nv 1e39 1 1\nv 2 2 2\nv 0 2 1\nvt 0 0\nvn 0 0 1\n"
                   "f 1/1/1 2/1/1 3/1/1\nf 4/1/1 5/1/1 6/1/1\nf 1/1/1 5/1/1 6/1/1\n")
    for spec in (("mesh_arrays", *nan_mesh(), ("diffuse", (1, 1, 1))), ("mesh", str(obj), ("diffuse", (1, 1, 1)))):
        sc = rt.Scene([spec])
        nodes, tris, _ = sc.flat_mesh(0)
        T = len(tris)
        assert T >= 2 and len(nodes) == 2 * T - 1 and nodes["escape"][0] == len(nodes)
        assert sorted(nodes["tri"][nodes["tri"] >= 0].tolist()) == list(range(T))
        corners = np.concatenate([tris["p0"], tris["p1"], tris["p2"]])
        assert not np.isfinite(corners).all()


# ---- GPU: primitives against the reference ---------------------------------------------------------------------
def _kat(rt, gpu, kind, rays, prims, width):
    prims = np.ascontiguousarray(prims, F).reshape(-1, width)
    n = len(prims)
    flags = np.zeros(n, np.int32)
    out7 = np.zeros((n, 7), F)
    rp = None if rays is None else np.ascontiguousarray(rays, F).ctypes.data
    assert rt.load_library().rt_gpu_kat(gpu.handle, kind, rp, prims.ctypes.data, width, n, flags.ctypes.data, out7.ctypes.data) == 0
    return flags, out7


def _tag_mismatch(tags, ok):
    return sorted(set(tags[~ok].tolist()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PRIMS))
def test_primitive_edges_bit_exact(rt, gpu, ref, name):
    """Every primitive at its edges == the reference, flags and all seven outputs.  For the slab test the hook also
    runs slab_fast wherever the walks run it (all axes enabled, finite ray, finite box) and turns a disagreement with
    slab_general into a mismatch here: on every finite box of the set the two agree."""
    kind, width, gen = PRIMS[name]
    rays, prims, tags = gen()
    f, o = _kat(rt, gpu, kind, rays, prims, width)
    rf, ro = getattr(ref, REF_FN[name])(rays, prims)
    ok_f = f == rf
    assert ok_f.all(), f"{name}: acceptance differs on {_tag_mismatch(tags, ok_f)}"
    if name == "slab":
        o, ro = o[:, 0], ro
        ok = (np.isnan(o) == np.isnan(ro)) & ((o.view(np.uint32) == ro.view(np.uint32)) | np.isnan(o))
    else:
        ok = ((np.isnan(o) == np.isnan(ro)) & ((o.view(np.uint32) == ro.view(np.uint32)) | np.isnan(o))).all(1)
    assert ok.all(), f"{name}: outputs differ on {_tag_mismatch(tags, ok)}"
    assert 0 < f.sum() < len(f)


@pytest.mark.gpu
def test_qrsqrt_and_barycentric_edges_bit_exact(rt, gpu, ref):
    x = scalar_edges()
    _, o = _kat(rt, gpu, 5, None, x, 1)
    assert same_bits(o[:, 0], ref.kat_qrsqrt(x))
    pabc, _ = barycentric_cases()
    _, o = _kat(rt, gpu, 6, None, pabc, 12)
    assert same_bits(o[:, :3], ref.kat_barycentric(pabc))


# ---- GPU: texture sampling on small and odd-sized textures ------------------------------------------------------------
def _textures():
    """1x1, 1xN, Nx1, 2x2 and odd-sized images, each a distinct constant or gradient: a tap from a neighbouring atlas
    rectangle shows up as a wrong colour."""
    out = []
    for k, (h, w, grad) in enumerate(((1, 1, False), (1, 7, True), (5, 1, True), (2, 2, True), (3, 5, False), (7, 3, True))):
        img = np.empty((h, w, 4), F)
        img[...] = np.array([k + 1, 10 * (k + 1), 0.5, 1], F)
        if grad:
            img[..., 2] = (np.arange(h)[:, None] * 100 + np.arange(w)[None, :] + 1).astype(F)
        out.append(img)
    return out


def _uv_edges():
    v = [F(0), F(-0.0), F(1), F(-1), F(2), F(-3), F(0.5), down(F(1)), up(F(-1)), F(1) - F(2.0) ** -24, -DENORM, DENORM,
         F(2.0) ** 23, F(2.0) ** 23 + F(1), -F(2.0) ** 23, F(2.0) ** 24 + F(2), F(1e30), -F(1e30), INF, -INF, NAN]
    g = np.array(v, F)
    return np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)


class _TexturedScene:
    """A one-triangle mesh with the images of _textures() as its texture slots, as a scene description."""

    def __init__(self, rt, images):
        A = rt._abi
        self.sc = rt.Scene([("mesh_arrays", [[0, 0, 0], [1, 0, 0], [0, 1, 0]], [[0, 1, 2]], ("diffuse", (1, 1, 1)))])
        d = self.sc.desc.contents
        self.images = [np.ascontiguousarray(im) for im in images]
        self.texs = (A.rt_texture * len(images))()
        for k, im in enumerate(self.images):
            self.texs[k].rgba = im.ctypes.data_as(C.POINTER(C.c_float))
            self.texs[k].width, self.texs[k].height = im.shape[1], im.shape[0]
        self.meshes = (A.rt_mesh * 1)()
        C.memmove(self.meshes, d.meshes, C.sizeof(A.rt_mesh))
        self.meshes[0].textures, self.meshes[0].num_textures = self.texs, len(images)
        self.desc = A.rt_scene_desc()
        C.memmove(C.byref(self.desc), C.byref(d), C.sizeof(self.desc))
        self.desc.meshes = self.meshes


def _kat_texture(rt, ctx, k, uv):
    out = np.zeros((len(uv), 4), F)
    assert rt.load_library().rt_gpu_kat_texture(ctx.handle, k, uv.ctypes.data, len(uv), out.ctypes.data) == 0
    return out


@pytest.mark.gpu
def test_texture_sample_edges(rt, port):
    """RTexture::Sample at integer, signed-zero, just-below-one, denormal, huge, infinite and NaN uv on 1x1, 1xN,
    Nx1, 2x2 and odd-sized textures == the restatement (which clamps the texel indices where the reference would read
    outside the image: the documented divergence for NaN / infinite uv); then float texels -0, denormals, +-inf, NaN
    and FLT_MAX written with rt_gpu_update_texture are sampled as the restatement samples the same array."""
    import torch
    images = _textures()
    ts = _TexturedScene(rt, images)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(C.pointer(ts.desc))
        uv = _uv_edges()
        for k, im in enumerate(images):
            assert same_bits(_kat_texture(rt, ctx, k, uv), port.kat_texture_sample(im, uv)), im.shape
        special = np.array([-0.0, 1e-40, -1e-40, np.inf, -np.inf, np.nan, FMAX, -FMAX, 1.5, TINY, -TINY, 2.0 ** -149], F)
        for k in (4, 5):
            h, w = images[k].shape[:2]
            tex = np.resize(special, (h, w, 4)).astype(F)
            tex[0, 0] = [-0.0, 1e-40, np.inf, np.nan]
            ctx.update_texture(0, k, torch.from_numpy(tex).to("cuda:0"))
            torch.cuda.synchronize()
            assert ctx.read_texture(0, k).tobytes() == tex.tobytes()
            got = _kat_texture(rt, ctx, k, uv)
            assert same_bits(got, port.kat_texture_sample(tex, uv)), k
        # the untouched images are still sampled as uploaded
        for k in (0, 1, 2, 3):
            assert same_bits(_kat_texture(rt, ctx, k, uv), port.kat_texture_sample(images[k], uv))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_texture_sample_edges_against_reference(rt, gpu, ref, data_dir):
    """Finite edge uv on the uploaded unitychan textures == the reference itself (inside the image it reads there)."""
    import scenes
    spec = scenes.c3_unitychan(data_dir)
    gpu.upload_scene(rt.Scene(spec))
    rs = ref.build_scene(spec)
    uv = _uv_edges()
    uv = uv[np.isfinite(uv).all(1)]
    k = 0
    for slot in range(ref.mesh_counts(rs, 0)[4]):
        if ref.mesh_texture(rs, 0, slot) is None:
            continue
        assert same_bits(_kat_texture(rt, gpu, k, uv), ref.kat_texture_sample(rs, 0, slot, uv)), slot
        k += 1
    assert k > 0
    ref.free_scene(rs)


# ---- GPU: boundary meshes through every walk kernel -------------------------------------------------------------------
def _boundary_meshes(scale):
    """Meshes at the edges the walks see: signed-zero coordinates, denormal offsets, duplicate and coincident triangles,
    flat meshes on each axis (flat boxes), at coordinate scale `scale`."""
    s = F(scale)
    out = []
    q = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0]], F)
    # signed zeros: +0 and -0 on every axis, the same position
    pz = np.array([[0.0, -0.0, 0.0], [1, 0, -0.0], [-0.0, 1, 0.0], [0, 0, -0.0], [-0.0, -0.0, 1], [1, -0.0, 1]], F) * s
    out.append((pz, np.array([[0, 1, 2], [3, 2, 1], [0, 4, 1], [3, 5, 2]], np.int32)))
    # denormal offsets of a unit grid
    g = np.array([[x, y, 0] for x in range(3) for y in range(3)], F) * s
    g[:, 2] = np.array([0, DENORM, -DENORM, F(1e-45), 0, -F(1e-45), DENORM * 3, 0, -DENORM], F)
    idx = [[3 * x + y, 3 * x + y + 3, 3 * x + y + 1] for x in range(2) for y in range(2)]
    out.append((g, np.array(idx, np.int32)))
    # duplicate and coincident triangles (same corners, other orders; and a copy of the points)
    t = np.concatenate([q, q], 0) * s + np.array([0, 0, 2], F) * s
    out.append((t, np.array([[0, 1, 2], [0, 1, 2], [1, 2, 0], [4, 5, 6], [2, 3, 0], [6, 7, 4]], np.int32)))
    # flat on x, on y, on z
    for axis in range(3):
        p = np.array([[a, b] for a in range(4) for b in range(4)], F) * s / F(3)
        p3 = np.insert(p, axis, F(0.5) * s, axis=1).astype(F) + F(3) * s * np.eye(3, dtype=F)[(axis + 1) % 3]
        idx = [[4 * a + b, 4 * a + b + 4, 4 * a + b + 1] for a in range(3) for b in range(3)]
        idx += [[4 * a + b + 1, 4 * a + b + 4, 4 * a + b + 5] for a in range(3) for b in range(3)]
        out.append((p3.astype(F), np.array(idx, np.int32)))
    return out


def _boundary_scene(rt, scale):
    return rt.Scene([("mesh_arrays", p, i, ("diffuse", (1, 1, 1))) for p, i in _boundary_meshes(scale)])


def _boundary_rays(sc, scale, seed=0):
    """Rays through vertices and edge midpoints, origins on node-box planes, direction components at the FLT_EPSILON
    cut-off (and one float either side), signed zeros in the direction."""
    rng = np.random.default_rng(seed)
    s = F(scale)
    rays = []
    d = sc.desc.contents
    for m in range(d.num_meshes):
        nodes, tris, _ = sc.flat_mesh(m)
        corners = np.concatenate([tris["p0"], tris["p1"], tris["p2"], (tris["p0"] + tris["p1"]) * F(0.5)])
        for p in corners:
            o = (p + rng.normal(size=3).astype(F) * s).astype(F)
            rays.append([*o, *(p - o), F(3)])
            o = (p + (rng.normal(size=3) * [0.5, 0.5, 0.5] + [0, 0, 2.5]).astype(F) * s).astype(F)   # from the front
            rays.append([*o, *(p - o), F(3)])
        for nd in nodes:
            for face in range(6):
                o = ((nd["bmin"] + nd["bmax"]) * F(0.5)).astype(F)
                o[face % 3] = (nd["bmin"] if face < 3 else nd["bmax"])[face % 3]
                for dd in (rng.normal(size=3).astype(F), -np.eye(3, dtype=F)[face % 3], np.eye(3, dtype=F)[face % 3]):
                    rays.append([*o, *dd, F(10) * s])
        centre = ((nodes[0]["bmin"] + nodes[0]["bmax"]) * F(0.5)).astype(F)
        for v in (EPS, down(EPS), up(EPS), -EPS, F(0), F(-0.0), DENORM):
            for axis in range(3):
                for _ in range(3):
                    o = (centre + rng.normal(size=3).astype(F) * s).astype(F)
                    dd = (centre - o).astype(F)
                    dd /= F(np.linalg.norm(dd))
                    dd[axis] = v
                    rays.append([*o, *dd, F(20) * s])
    return np.array(rays, F)


WALK_VARIANTS = (dict(), dict(RT_LONG_LIMIT="8", RT_SMALL_ROUND="0", RT_THIN_COUNT="0"))
KNOBS = ("RT_LONG_LIMIT", "RT_SMALL_ROUND", "RT_THIN_COUNT", "RT_PACKET_ROUNDS")


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 1e4])
@pytest.mark.parametrize("traverse", ["exact", "culled"])
def test_boundary_meshes_through_every_walk(rt, port, monkeypatch, scale, traverse):
    """Accepted boundary meshes: query_rays (the production wavefront walks) and trace_rays (the hook's walk) == the
    restatement's trace_rays bit for bit (shape, triangle, all 11 hit fields); PRIMARY renders (packets form in the
    camera round) == the restatement's ids and Distance bits; for every walk variant (packets, long walks after 8
    steps) and, exact, the same slab and triangle test counts."""
    import torch
    sc = _boundary_scene(rt, scale)
    d = sc.desc.contents
    d.eye[0], d.eye[1], d.eye[2] = F(1.5 * scale), F(1.5 * scale), F(5 * scale)
    d.ray_distance = F(100 * scale)
    rays = _boundary_rays(sc, scale)
    ws, wt, wh = port.trace_rays(sc.desc, rays)
    assert (ws >= 0).sum() > 50
    W, H = 160, 96
    p = rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=rt.RT_TRAVERSE_EXACT)
    want = port.render(sc.desc, p, nthreads=os.cpu_count() or 1, want_primary=True)
    trav = rt.RT_TRAVERSE_EXACT if traverse == "exact" else rt.RT_TRAVERSE_CULLED
    counts = None
    for env in WALK_VARIANTS:
        for k in KNOBS:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ctx = rt.GpuContext(0)
        try:
            ctx.upload_scene(sc)
            ctx.reset_counters()
            q = ctx.query_rays(torch.from_numpy(rays).to("cuda:0"), traverse=trav)
            torch.cuda.synchronize()
            ctx.synchronize()
            c = ctx.counters()
            assert np.array_equal(q["shape"].cpu().numpy(), ws), env
            assert np.array_equal(q["tri"].cpu().numpy(), wt), env
            assert same_bits(q["hit"].cpu().numpy(), wh), env
            gs, gt, gh = ctx.trace_rays(rays, traverse=trav)
            assert np.array_equal(gs, ws) and np.array_equal(gt, wt) and same_bits(gh, wh), env
            if traverse == "exact":
                now = (c["node_tests"], c["tri_tests"])
                assert counts is None or now == counts, env
                counts = now
            pp = rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=trav)
            ctx.reset_accum(W, H)
            ctx.render_tile(pp)
            ids = ctx.readback(rt.RT_READ_PRIMARY_IDS_I32X2, W, H)
            dist = ctx.readback(rt.RT_READ_PRIMARY_DIST_F32, W, H)
            assert np.array_equal(ids.reshape(-1, 2), want["ids"].reshape(-1, 2)), env
            assert same_bits(dist.reshape(-1), want["dist"].reshape(-1)), env
        finally:
            ctx.close()


# ---- GPU: refusals of non-finite geometry --------------------------------------------------------------------------
# tilted triangles: a triangle in a plane z = const has flat leaf boxes, which the reference's slab test never enters
GOOD_POINTS = np.array([[-1, -1, -3], [1, -1, -3.5], [0, 1, -3.2], [-2, -2, -4], [2, -2, -4.5], [0, 2, -4.2], [0, 0, 0]], F)


def _good_scene(rt):
    return rt.Scene([("mesh_arrays", GOOD_POINTS[:6], np.array([[0, 1, 2], [3, 4, 5]], np.int32), ("diffuse", (1, 1, 1))),
                     ("sphere", (0.5, 0.5, -6), 1.0, ("diffuse", (1, 0.5, 0.2)))])


def _renders_as_restatement(rt, port, ctx, sc):
    rng = np.random.default_rng(0)
    o = np.zeros((500, 3), F)
    dd = (rng.normal(size=(500, 3)) * [0.4, 0.4, 0.1] + [0, 0, -1]).astype(F)
    rays = np.concatenate([o, dd, np.full((500, 1), 50, F)], 1)
    ws, wt, wh = port.trace_rays(sc.desc, rays)
    for trav in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        gs, gt, gh = ctx.trace_rays(rays, traverse=trav)
        assert np.array_equal(gs, ws) and np.array_equal(gt, wt) and same_bits(gh, wh)
    assert (ws == 0).any() and (ws == 1).any()


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["nan", "inf", "-inf"])
def test_upload_refuses_non_finite_corner(rt, port, bad):
    ctx = rt.GpuContext(0)
    try:
        pts, idx = nan_mesh(F(bad))
        sc = rt.Scene([("sphere", (0, 0, -5), 1.0, ("diffuse", (1, 1, 1))), ("mesh_arrays", pts, idx, ("diffuse", (1, 1, 1)))])
        with pytest.raises(rt.RtError, match="mesh 0: non-finite"):
            ctx.upload_scene(sc)
        good = _good_scene(rt)
        ctx.upload_scene(good)
        _renders_as_restatement(rt, port, ctx, good)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_upload_refuses_obj_with_nan_and_overflow(rt, port, tmp_path):
    """The loader reads `nan` and `1e39` (inf) with strtof; the upload refuses the mesh (the inf reaches the node bounds
    too, which are checked first)."""
    for bad in ("nan", "1e39"):
        text = f"v 0 0 -3\nv 1 0 -3\nv {bad} 1 -3\nvt 0 0\nvn 0 0 1\nf 1/1/1 2/1/1 3/1/1\n"
        obj = tmp_path / "bad.obj"
        obj.write_text(text)
        ctx = rt.GpuContext(0)
        try:
            with pytest.raises(rt.RtError, match="mesh 0: non-finite"):
                ctx.upload_scene(rt.Scene([("mesh", str(obj), ("diffuse", (1, 1, 1)))]))
            good = _good_scene(rt)
            ctx.upload_scene(good)
            _renders_as_restatement(rt, port, ctx, good)
        finally:
            ctx.close()


@pytest.mark.gpu
def test_upload_refuses_nan_node_bound(rt, port):
    """A hand-made description whose corners are finite but one node bound is NaN (the host layer never emits one)."""
    sc = _good_scene(rt)
    node = sc.desc.contents.meshes[0].nodes[0]
    ctx = rt.GpuContext(0)
    try:
        for field, c in (("bmin", 0), ("bmax", 0), ("bmax", 2)):
            keep = getattr(node, field)[c]
            getattr(node, field)[c] = float("nan")
            try:
                with pytest.raises(rt.RtError, match="mesh 0: non-finite BVH node bound"):
                    ctx.upload_scene(sc)
            finally:
                getattr(node, field)[c] = keep
        ctx.upload_scene(sc)
        _renders_as_restatement(rt, port, ctx, sc)
    finally:
        ctx.close()


def _mesh_bytes(ctx, mesh=0):
    nodes, tris, shade, bounds, scale = ctx.read_mesh(mesh)
    return nodes.tobytes() + tris.tobytes() + shade.tobytes() + bounds.tobytes() + scale.tobytes()


@pytest.mark.gpu
def test_mesh_edits_refuse_non_finite_points(rt, port):
    """update_mesh and replace_mesh with a NaN point, used by a triangle or by none: RT_ERR_INVALID naming it, and the
    mesh as the device holds it unchanged byte for byte; a refit reports status 16 (17 with a bad point index too),
    publishes nothing, and a following good refit publishes."""
    import torch
    sc = _good_scene(rt)
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        before = _mesh_bytes(ctx)
        pts = GOOD_POINTS.copy()
        idx = torch.from_numpy(np.array([[0, 1, 2], [3, 4, 5]], np.int32)).to("cuda:0")
        for row in (1, 6):                                  # a used point, and the point no triangle uses
            for bad in (NAN, INF):
                p = pts.copy()
                p[row, 1] = bad
                dp = torch.from_numpy(p).to("cuda:0")
                with pytest.raises(rt.RtError, match="rt_gpu_update_mesh: non-finite point"):
                    ctx.update_mesh(0, dp, idx)
                assert _mesh_bytes(ctx) == before
                with pytest.raises(rt.RtError, match="rt_gpu_replace_mesh: non-finite point"):
                    ctx.replace_mesh(0, dp, idx[:1].contiguous())
                assert _mesh_bytes(ctx) == before
                st = ctx.refit_mesh(0, dp, idx)
                assert int(st.cpu()[0]) == 16
                assert _mesh_bytes(ctx) == before
                bad_idx = torch.from_numpy(np.array([[0, 1, 2], [3, 4, 99]], np.int32)).to("cuda:0")
                st = ctx.refit_mesh(0, dp, bad_idx)
                assert int(st.cpu()[0]) == 17
                assert _mesh_bytes(ctx) == before
        _renders_as_restatement(rt, port, ctx, sc)
        moved = pts.copy()
        moved[:, 0] += F(0.25)
        st = ctx.refit_mesh(0, torch.from_numpy(moved).to("cuda:0"), idx)
        assert int(st.cpu()[0]) == 0
        assert _mesh_bytes(ctx) != before
        fresh = rt.Scene([("mesh_arrays", moved, np.array([[0, 1, 2], [3, 4, 5]], np.int32), ("diffuse", (1, 1, 1))),
                          ("sphere", (0.5, 0.5, -6), 1.0, ("diffuse", (1, 0.5, 0.2)))])
        _renders_as_restatement(rt, port, ctx, fresh)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_build_bvh_refuses_non_finite_points(rt, gpu):
    pts, idx = nan_mesh()
    for bad in (NAN, INF, -INF):
        p = pts.copy()
        p[4, 1] = bad
        with pytest.raises(rt.RtError, match="non-finite point"):
            gpu.build_bvh(p, idx)
    p = np.concatenate([pts, [[np.nan, 0, 0]]]).astype(F)       # a point no triangle uses
    p[4, 1] = 1
    with pytest.raises(rt.RtError, match="non-finite point"):
        gpu.build_bvh(p, idx)
    nodes, tris, _, _ = gpu.build_bvh(p[:-1], idx)
    assert len(nodes) == 3 and len(tris) == 2
