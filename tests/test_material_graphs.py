"""Material graphs (rt_material arrays) against the restatement: generated trees of every class up to the Combine nesting
the device holds (RT_MAX_MATERIAL_DEPTH = 8), nodes shared by index, paths that run the whole bounce budget, and the
upload's refusal of graphs material_eval cannot compute (cycles, deeper nesting, shape materials below -1).

No test renders, queries or hands to the restatement a graph with a cycle: the device would loop and the restatement
would recurse without end.  Graphs that must be refused are uploaded on a context of their own, closed in `finally`, so
that no such scene stays resident; an upload that unexpectedly succeeds fails the test before anything is rendered."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import same_bits
from test_radiance_queries import counted, radiance, restatement  # noqa: F401  (restatement: fixture)
from test_ray_queries import pinhole_rays, random_rays

MAX_COMBINES = 8            # RT_MAX_MATERIAL_DEPTH, rt_device.cuh
PATH, PREVIEW = 0, 1
TRAVERSALS = (0, 1)         # RT_TRAVERSE_EXACT, RT_TRAVERSE_CULLED
DIFFUSE, CHECKER, REFLECTIVE, EMISSIVE, BLEND, COMBINE, NULL = range(7)
FLT_EPS = np.float32(1.1920929e-07)
NAN = float("nan")

# ---------------------------------------------------------------------------------------------------
# generated trees (material specs of raytracerwin_b200.Scene)
# ---------------------------------------------------------------------------------------------------
# Blend factors: the ends, one ulp-scale step inside them, NaN (rng_random() > NaN is false: always B), and values the
# host layer clamps to [0, 1].  Checker sizes: 0 and 1e-30 fall back to 1, a negative size flips the pattern, 1e30
# leaves a reciprocal of 1e-30.
BLEND_FACTORS = (0.0, 1.0, 1e-7, 1.0 - 1e-7, NAN, -0.5, 1.5, 0.5, 0.25)
CHECKER_SIZES = (5.0, 0.0, -3.0, 1e-30, 1e30)
LEVELS = (0.0, 0.25, 0.5, 0.75, 1.0)


def _rgb(rng, zero_ok=True):
    c = tuple(float(x) for x in rng.choice(LEVELS[1:], 3))
    return (0.0, 0.0, 0.0) if zero_ok and rng.random() < 0.2 else c


def random_leaf(rng, fuzzy):
    k = int(rng.integers(5))
    if k == 0:
        return ("diffuse", _rgb(rng))
    if k == 1:
        return ("checker", _rgb(rng), float(rng.choice(CHECKER_SIZES)))
    if k == 2:
        return ("reflective", _rgb(rng), float(rng.choice((0.05, 0.3))) if fuzzy else 0.0)
    if k == 3:
        return ("emissive", _rgb(rng))              # zero emission included
    return ("null",)


def random_tree(rng, combines, fuzzy, blends=2):
    """A tree whose deepest path passes exactly `combines` Combine nodes, with up to `blends` Blends on a path."""
    if blends > 0 and rng.random() < 0.3:
        return ("blend", random_tree(rng, combines, fuzzy, blends - 1),
                random_tree(rng, int(rng.integers(0, combines + 1)), fuzzy, blends - 1), float(rng.choice(BLEND_FACTORS)))
    if combines == 0:
        return random_leaf(rng, fuzzy)
    deep = random_tree(rng, combines - 1, fuzzy, blends)
    other = random_tree(rng, int(rng.integers(0, min(combines, 3))), fuzzy, blends)
    return ("combine", deep, other) if rng.random() < 0.5 else ("combine", other, deep)


def chain(n, via, end=("emissive", (0.25, 0.5, 0.75)), blends=False):
    """n nested Combines through child_a ("a") or child_b ("b"), each adding a leaf of its own; with `blends`, a Blend
    between every two levels whose two children both continue the chain."""
    t = end
    for k in range(n):
        leaf = ("emissive", (0.0, 0.0, 0.25)) if k % 2 else ("reflective", (0.5, 0.5, 0.5), 0.0)
        if blends:
            t = ("blend", t, t, 0.5)
        t = ("combine", t, leaf) if via == "a" else ("combine", leaf, t)
    return t


def combine_depth(spec):
    k = spec[0]
    if k in ("blend", "combine"):
        return max(combine_depth(spec[1]), combine_depth(spec[2])) + (k == "combine")
    return 0


def generated_trees(seed, fuzzy=False, count=24):
    """Chains of exactly MAX_COMBINES through child_b, through child_a and across Blends, one random tree of every
    Combine depth 0..MAX_COMBINES, then random depths."""
    rng = np.random.default_rng(seed)
    trees = [chain(MAX_COMBINES, "b"), chain(MAX_COMBINES, "a"), chain(MAX_COMBINES, "b", blends=True)]
    trees += [random_tree(rng, d, fuzzy) for d in range(MAX_COMBINES + 1)]
    while len(trees) < count:
        trees.append(random_tree(rng, int(rng.integers(0, MAX_COMBINES + 1)), fuzzy))
    return trees


def shapes_with(mats, data_dir):
    """Sphere, capsule, plane, triangle, TorusKnot and unitychan (textures with varying alpha), materials in order."""
    return [("sphere", (1.2, 0.8, -1.0), 0.7, mats[0]),
            ("capsule", (-0.5, -1.2, 0.5), (0.8, -1.4, 1.0), 0.3, mats[1]),
            ("plane", (0.0, 1.0, 0.0), (0.0, -2.0, 0.0), mats[2]),
            ("triangle", (-2.5, -1.0, -2.0), (2.5, -1.0, -2.0), (0.0, 2.5, -2.5), mats[3]),
            ("mesh", os.path.join(data_dir, "TorusKnot.obj"), mats[4]),
            ("mesh", os.path.join(data_dir, "unitychan.obj"), mats[5])]


def generated_scenes(rt, data_dir, seed, fuzzy=False):
    trees = generated_trees(seed, fuzzy)
    for k in range(0, len(trees), 6):
        sc = rt.Scene(shapes_with(trees[k:k + 6], data_dir))
        sc.set_unit_vectors(seed=seed, count=1 << 18)
        yield sc


# ---------------------------------------------------------------------------------------------------
# graphs written straight into a scene's description
# ---------------------------------------------------------------------------------------------------
class Graph:
    """An rt_material array built node by node.  of(spec) flattens a spec as the host layer does (Checker: reciprocal of
    the size, 1 below FLT_EPSILON; Blend factor clamped to [0, 1]), except that the same spec OBJECT gives the same
    node (unless share=False): a subtree used twice is shared by index instead of copied."""

    def __init__(self, share=True):
        self.nodes, self._memo, self.share = [], {}, share

    def add(self, t, a=-1, b=-1, rgb=(0.0, 0.0, 0.0), scalar=0.0):
        self.nodes.append((t, a, b, tuple(rgb), float(scalar)))
        return len(self.nodes) - 1

    def of(self, spec):
        if self.share and id(spec) in self._memo:
            return self._memo[id(spec)][0]
        k = spec[0]
        if k == "blend":
            a, b = self.of(spec[1]), self.of(spec[2])
            f = np.float32(spec[3])
            i = self.add(BLEND, a, b, scalar=f if np.isnan(f) else min(max(f, np.float32(0)), np.float32(1)))
        elif k == "combine":
            a, b = self.of(spec[1]), self.of(spec[2])
            i = self.add(COMBINE, a, b)
        elif k == "checker":
            size = np.float32(spec[2])
            i = self.add(CHECKER, rgb=spec[1], scalar=1.0 if abs(size) < FLT_EPS else np.float32(1) / size)
        elif k == "null":
            i = self.add(NULL)
        else:
            i = self.add({"diffuse": DIFFUSE, "reflective": REFLECTIVE, "emissive": EMISSIVE}[k], rgb=spec[1],
                         scalar=spec[2] if k == "reflective" else 0.0)
        self._memo[id(spec)] = (i, spec)          # the spec stays referenced, so its id is not reused
        return i


def set_materials(rt, sc, nodes, roots):
    """Points Scene `sc`'s description at the material array `nodes` ((type, a, b, rgb, scalar) each), shape i at node
    roots[i].  The array lives as long as the scene (the description is only rebuilt when the scene changes)."""
    abi = rt._abi
    arr = (abi.rt_material * max(len(nodes), 1))()
    for k, (t, a, b, rgb, s) in enumerate(nodes):
        arr[k] = abi.rt_material(t, a, b, abi.f3(*rgb), s)
    d = sc.desc.contents
    d.materials, d.num_materials = C.cast(arr, C.POINTER(abi.rt_material)), len(nodes)
    for i, r in enumerate(roots):
        d.shapes[i].material = r
    sc._materials = arr
    return sc


def desc_nodes(sc):
    d = sc.desc.contents
    return [(m.type, m.child_a, m.child_b, tuple(m.rgb), m.scalar) for m in d.materials[:d.num_materials]]


def upload_allowed(nodes, shape_materials):
    """The upload's rule, stated independently: child indices in range, every shape material in [-1, n), and from every
    node no cycle and at most MAX_COMBINES Combines on any path down to a leaf (recursive, for small graphs)."""
    n = len(nodes)
    if any(m < -1 or m >= n for m in shape_materials):
        return False
    depth = {}

    def deepest(i, path):
        if i in path:
            raise RecursionError
        if i not in depth:
            t, a, b = nodes[i][:3]
            if t in (BLEND, COMBINE):
                depth[i] = max(deepest(a, path | {i}), deepest(b, path | {i})) + (t == COMBINE)
            else:
                depth[i] = 0
        return depth[i]

    for t, a, b in (nd[:3] for nd in nodes):
        if t in (BLEND, COMBINE) and not (0 <= a < n and 0 <= b < n):
            return False
    try:
        return all(deepest(i, frozenset()) <= MAX_COMBINES for i in range(n))
    except RecursionError:
        return False


# ---------------------------------------------------------------------------------------------------
# without a GPU: the generator, the host layer's flattening, shared nodes and the reference
# ---------------------------------------------------------------------------------------------------
def test_generated_trees_reach_every_class_and_value(rt, data_dir):
    trees = generated_trees(1) + generated_trees(2)
    assert [combine_depth(t) for t in trees[:12]] == [MAX_COMBINES] * 3 + list(range(MAX_COMBINES + 1))
    assert max(combine_depth(t) for t in trees) == MAX_COMBINES
    nodes = []
    for sc in list(generated_scenes(rt, data_dir, 1)) + list(generated_scenes(rt, data_dir, 2)):
        nodes += desc_nodes(sc)
    types = {t for t, *_ in nodes}
    assert types == set(range(7))
    blend = np.float32([s for t, _, _, _, s in nodes if t == BLEND])
    # NaN reaches the description unclamped; -0.5 and 1.5 arrive as 0 and 1
    assert np.isnan(blend).any()
    assert set(blend[~np.isnan(blend)].tolist()) == set(np.float32([0.0, 1.0, 1e-7, 1.0 - 1e-7, 0.5, 0.25]).tolist())
    checker = set(np.float32([s for t, _, _, _, s in nodes if t == CHECKER]).tolist())
    assert checker == set(np.float32([0.2, 1.0, np.float32(1) / np.float32(-3.0), 1e-30]).tolist())
    emit = [rgb for t, _, _, rgb, _ in nodes if t == EMISSIVE]
    assert any(rgb == (0.0, 0.0, 0.0) for rgb in emit) and any(rgb != (0.0, 0.0, 0.0) for rgb in emit)
    # Graph.of flattens a tree exactly as the host layer does
    for sc, k in zip(generated_scenes(rt, data_dir, 3), range(0, 24, 6)):
        g = Graph(share=False)
        roots = [g.of(t) for t in generated_trees(3)[k:k + 6]]
        assert [sc.desc.contents.shapes[i].material for i in range(6)] == roots
        got, want = desc_nodes(sc), g.nodes
        assert [n[:3] for n in got] == [n[:3] for n in want]
        assert same_bits([n[3] + (n[4],) for n in got], [n[3] + (n[4],) for n in want])


def shared_graph_specs():
    """Shape materials in which one Combine subtree is used by two shapes and twice under one parent."""
    sub = ("combine", ("blend", ("reflective", (0.75, 0.75, 0.5), 0.0), ("diffuse", (0.5, 1.0, 0.25)), 0.5),
           ("emissive", (0.25, 0.0, 0.5)))
    two = ("combine", sub, ("blend", sub, ("checker", (1.0, 0.5, 0.5), 5.0), 0.25))
    return [two, sub, ("combine", ("null",), two), ("reflective", (0.5, 0.5, 0.75), 0.0), sub, two]


def shared_scenes(rt, data_dir):
    """(the graph with shared nodes, its tree expansion built through the host layer)"""
    specs = shared_graph_specs()
    tree = rt.Scene(shapes_with(specs, data_dir))
    tree.set_unit_vectors(seed=4, count=1 << 18)
    dag = rt.Scene(shapes_with([("null",)] * 6, data_dir))
    dag.set_unit_vectors(seed=4, count=1 << 18)
    g = Graph()
    roots = [g.of(s) for s in specs]
    assert len(g.nodes) < tree.desc.contents.num_materials
    return set_materials(rt, dag, g.nodes, roots), tree


def test_shared_nodes_equal_the_tree_expansion_in_the_restatement(rt, port, restatement, data_dir):
    dag, tree = shared_scenes(rt, data_dir)
    W, H = 96, 72
    for mode, bounce in ((PATH, 1), (PATH, 3), (PATH, 10), (PREVIEW, 10)):
        p = rt.make_params(W, H, mode=mode, max_bounce=bounce, antialias=1, seed=3, traverse=rt.RT_TRAVERSE_EXACT)
        a, b = port.render(dag.desc, p, nthreads=os.cpu_count() or 1), port.render(tree.desc, p, nthreads=os.cpu_count() or 1)
        key = "preview" if mode == PREVIEW else "accum"
        assert same_bits(a[key], b[key]), (mode, bounce)
        assert a["counters"]["rays"] == b["counters"]["rays"]
    rays = random_rays(4000, 8)
    for mode, bounce in ((PATH, 10), (PREVIEW, 10)):
        a = restatement.radiance_rays(dag.desc, rays, mode, bounce, 5, 1, np.arange(len(rays)), 0)
        b = restatement.radiance_rays(tree.desc, rays, mode, bounce, 5, 1, np.arange(len(rays)), 0)
        assert same_bits(a[0], b[0]) and a[1] == b[1]


def test_restatement_equals_the_reference_on_generated_trees(rt, port, data_dir):
    from oracle import bindings
    if not bindings.ref_available():
        pytest.skip("oracle/_ref/libref_oracle.so not built")
    ref = bindings.RefOracle()
    ref.init_unit_vectors(2)
    W, H = 64, 48
    trees = generated_trees(6)
    for k in range(0, len(trees), 6):
        spec = shapes_with(trees[k:k + 6], data_dir)
        sc = rt.Scene(spec)
        sc.set_unit_vectors(seed=2, count=0)
        rs = ref.build_scene(spec)
        for mode, bounce in ((PATH, 3), (PATH, 10), (PREVIEW, 10)):
            p = rt.make_params(W, H, mode=mode, max_bounce=bounce, antialias=1, seed=7, traverse=rt.RT_TRAVERSE_EXACT)
            o = port.render(sc.desc, p, nthreads=8)
            r = ref.render(rs, W, H, mode=mode, max_bounce=bounce, antialias=1, seed=7, nthreads=8)
            assert same_bits((o["preview"] if mode == PREVIEW else o["accum"])[..., :3], r["accum"][..., :3]), (k, mode)
        ref.free_scene(rs)


# ---------------------------------------------------------------------------------------------------
# on the GPU, bit for bit
# ---------------------------------------------------------------------------------------------------
def render_gpu(rt, gpu, W, H, tr, **kw):
    """One render_tile call after a reset: (image, rays counted); the image is the preview colour in RT_MODE_PREVIEW."""
    gpu.reset_accum(W, H)
    _, c = counted(gpu, lambda: gpu.render_tile(rt.make_params(W, H, traverse=tr, **kw)))
    prev = kw.get("mode") == PREVIEW
    img = gpu.readback(rt.RT_READ_PREVIEW_RGBA_F32 if prev else rt.RT_READ_ACCUM_RGBN_F32, W, H)
    return (img[..., :3] if prev else img), c["rays"]


def render_port(rt, port, sc, W, H, **kw):
    """The restatement's render of the same call: (image, rays counted)."""
    o = port.render(sc.desc, rt.make_params(W, H, **kw), nthreads=os.cpu_count() or 1)
    return (o["preview"][..., :3] if kw.get("mode") == PREVIEW else o["accum"]), o["counters"]["rays"]


@pytest.mark.gpu
def test_generated_trees_bit_exact(rt, gpu, port, restatement, data_dir):
    W, H = 96, 72
    rays = np.concatenate([pinhole_rays(96, 64, True), random_rays(8000, 17)])
    streams = 100 + np.arange(len(rays), dtype=np.uint32)
    for k, sc in enumerate(generated_scenes(rt, data_dir, 11)):
        gpu.upload_scene(sc)
        for mode, bounce in ((PATH, 1), (PATH, 3), (PATH, 10), (PREVIEW, 10)):
            kw = dict(mode=mode, max_bounce=bounce, antialias=1, seed=k + 1)
            want, wn = render_port(rt, port, sc, W, H, **kw)
            for tr in TRAVERSALS:
                got, n = render_gpu(rt, gpu, W, H, tr, **kw)
                assert same_bits(got, want), (k, mode, bounce, tr)
                assert n == wn, (k, mode, bounce, tr)
            want, wc = restatement.radiance_rays(sc.desc, rays, mode, bounce, 9, 2, streams, 0)
            for tr in TRAVERSALS:
                got, c = counted(gpu, lambda: radiance(gpu, rays, mode=mode, max_bounce=bounce, seed=9, sample=2,
                                                       rng_stream_base=100, traverse=tr))
                assert same_bits(got[:, :3], want), (k, mode, bounce, tr)
                assert c["rays"] == wc["rays"], (k, mode, bounce, tr)
            if mode == PATH and bounce == 10:
                assert wc["rays"] > 2 * len(rays)     # paths did bounce


@pytest.mark.gpu
def test_full_depth_paths(rt, gpu, port, restatement, data_dir):
    """Combine(Emissive, Reflective fuzz 0): Emissive is evaluated last, so the outgoing ray is the incoming one and a
    path that meets the sphere re-traces it until max_bounce = 32 segments (the unwinding stack full).  On unitychan a
    texel's alpha lets a re-traced path pass through after any number of segments (pass-through bits up to 31)."""
    loop = ("combine", ("emissive", (0.25, 0.125, 0.5)), ("reflective", (0.5, 0.75, 0.5), 0.0))
    sc = rt.Scene([("sphere", (1.5, 0.5, -1.0), 0.8, loop),
                   ("mesh", os.path.join(data_dir, "unitychan.obj"), loop),
                   ("plane", (0.0, 1.0, 0.0), (0.0, -2.0, 0.0), ("reflective", (0.75, 0.75, 0.75), 0.0))])
    gpu.upload_scene(sc)
    W, H = 160, 120
    want, wn = render_port(rt, port, sc, W, H, mode=PATH, max_bounce=32, antialias=1, seed=5)
    for tr in TRAVERSALS:
        got, n = render_gpu(rt, gpu, W, H, tr, mode=PATH, max_bounce=32, antialias=1, seed=5)
        assert same_bits(got, want), tr
        assert n == wn, tr
    rays = np.concatenate([pinhole_rays(W, H, True), random_rays(20_000, 23)])
    first = gpu.trace_rays(rays)[0]
    assert (first == 0).sum() > 100 and (first == 1).sum() > 100
    want, wc = restatement.radiance_rays(sc.desc, rays, PATH, 32, 3, 0, np.arange(len(rays)), 0)
    assert wc["rays"] >= 32 * (first == 0).sum()
    for tr in TRAVERSALS:
        got, c = counted(gpu, lambda: radiance(gpu, rays, mode=PATH, max_bounce=32, seed=3, traverse=tr))
        assert same_bits(got[:, :3], want), tr
        assert c["rays"] == wc["rays"], tr


@pytest.mark.gpu
def test_shared_subtrees(rt, gpu, port, restatement, data_dir):
    dag, tree = shared_scenes(rt, data_dir)
    W, H = 96, 72
    rays = random_rays(8000, 29)
    for mode, bounce in ((PATH, 3), (PATH, 10), (PREVIEW, 10)):
        kw = dict(mode=mode, max_bounce=bounce, seed=2)
        want, wc = restatement.radiance_rays(tree.desc, rays, mode, bounce, 1, 0, np.arange(len(rays)), 0)
        img, wn = render_port(rt, port, tree, W, H, **kw)
        for tr in TRAVERSALS:
            imgs = []
            for sc in (dag, tree):
                gpu.upload_scene(sc)
                got, n = render_gpu(rt, gpu, W, H, tr, **kw)
                assert same_bits(got, img) and n == wn, (mode, bounce, tr)
                imgs.append(got)
                got, c = counted(gpu, lambda: radiance(gpu, rays, mode=mode, max_bounce=bounce, seed=1, traverse=tr))
                assert same_bits(got[:, :3], want) and c["rays"] == wc["rays"], (mode, bounce, tr)
            assert same_bits(imgs[0], imgs[1])


@pytest.mark.gpu
def test_fuzzy_leaves_within_the_render_bar(rt, gpu, port, data_dir):
    """Fuzzy reflection calls sinf / cosf / acosf, whose CUDA and glibc results differ in the last ulp and can steer a
    path elsewhere: >= 99.9 % of pixels within 1e-4 and the image mean within 0.1 %.  A Combine adds the attenuation of
    both children, so radiance here reaches 1e5 and more, where one float ulp exceeds 1e-4: the tolerance is 1e-4
    relative to the colour above 1."""
    W, H = 128, 96
    for k, sc in enumerate(generated_scenes(rt, data_dir, 12, fuzzy=True)):
        gpu.upload_scene(sc)
        kw = dict(mode=PATH, max_bounce=10, antialias=1, pass_count=2, seed=k)
        got, n = render_gpu(rt, gpu, W, H, rt.RT_TRAVERSE_CULLED, **kw)
        want, wn = render_port(rt, port, sc, W, H, **kw)
        assert n == wn, k
        g, r = got[..., :3].reshape(-1, 3), want[..., :3].reshape(-1, 3)
        bad = (np.abs(g - r) > 1e-4 * np.maximum(1.0, np.abs(r))).any(1) | (np.isnan(g) != np.isnan(r)).any(1)
        assert bad.mean() <= 1e-3, (k, bad.mean())
        ok = np.isfinite(g).all(1) & np.isfinite(r).all(1)
        assert abs(g[ok].mean() - r[ok].mean()) <= 1e-3 * abs(r[ok].mean()), k


# ---------------------------------------------------------------------------------------------------
# graphs the upload refuses
# ---------------------------------------------------------------------------------------------------
def _two_spheres(rt):
    sc = rt.Scene([("sphere", (1.2, 0.8, -1.0), 0.7, ("null",)), ("sphere", (-1.4, 0.2, -0.5), 0.6, ("null",))])
    sc.set_unit_vectors(seed=0, count=1 << 16)
    return sc


def refused_graphs(rt):
    """{name: (scene, a word the error text must contain)}"""
    out = []
    for name, spec in (("depth 9 via child_b", chain(MAX_COMBINES + 1, "b")),
                       ("depth 9 via child_a", chain(MAX_COMBINES + 1, "a")),
                       ("depth 9 across Blends", chain(MAX_COMBINES + 1, "b", blends=True))):
        g = Graph()
        out.append((name, set_materials(rt, _two_spheres(rt), g.nodes, [g.of(spec), -1]), "Combine"))
    g = Graph()                                         # depth 9 under a node no shape uses
    g.of(chain(MAX_COMBINES + 1, "a"))
    out.append(("depth 9 unused", set_materials(rt, _two_spheres(rt), g.nodes, [g.of(("diffuse", (1, 1, 1))), -1]),
                "Combine"))
    g = Graph()
    leaf = g.add(EMISSIVE, rgb=(1, 1, 1))
    self_loop = g.add(BLEND, scalar=0.5)
    g.nodes[self_loop] = (BLEND, self_loop, self_loop, (0, 0, 0), 0.5)
    out.append(("Blend self-loop", set_materials(rt, _two_spheres(rt), g.nodes, [self_loop, leaf]), "cycle"))
    g = Graph()
    leaf = g.add(REFLECTIVE, rgb=(0.5, 0.5, 0.5))
    a = g.add(COMBINE, leaf, 2)
    g.add(COMBINE, a, leaf)
    out.append(("two-node Combine cycle", set_materials(rt, _two_spheres(rt), g.nodes, [a, leaf]), "cycle"))
    g = Graph()
    leaf = g.add(DIFFUSE, rgb=(1, 0.5, 0.25))
    b = g.add(BLEND, leaf, 3, scalar=0.5)               # 1 -> 3 -> 2 -> 1: reachable from no shape
    g.add(COMBINE, b, leaf)
    g.add(BLEND, 2, leaf, scalar=0.5)
    out.append(("cycle no shape reaches", set_materials(rt, _two_spheres(rt), g.nodes, [leaf, leaf]), "cycle"))
    g = Graph()
    leaf = g.add(EMISSIVE, rgb=(1, 1, 1))
    out.append(("shape material -2", set_materials(rt, _two_spheres(rt), g.nodes, [-2, leaf]), "material"))
    return {name: (sc, word) for name, sc, word in out}


REFUSED = ("depth 9 via child_b", "depth 9 via child_a", "depth 9 across Blends", "depth 9 unused", "Blend self-loop",
           "two-node Combine cycle", "cycle no shape reaches", "shape material -2")


@pytest.mark.gpu
@pytest.mark.parametrize("name", REFUSED)
def test_refused_graphs(rt, restatement, name):
    bad, words = refused_graphs(rt)[name]
    good = _two_spheres(rt)
    g = Graph()
    set_materials(rt, good, g.nodes, [g.of(chain(MAX_COMBINES, "b", blends=True)), g.of(chain(MAX_COMBINES, "a"))])
    rays = random_rays(4000, 31)
    ctx = rt.GpuContext(0)
    try:
        with pytest.raises(rt.RtError) as e:
            ctx.upload_scene(bad)
        assert words in str(e.value), (name, str(e.value))
        ctx.upload_scene(good)
        want, _ = restatement.radiance_rays(good.desc, rays, PATH, 10, 2, 0, np.arange(len(rays)), 0)
        assert same_bits(radiance(ctx, rays, max_bounce=10, seed=2)[:, :3], want), name
    finally:
        ctx.close()


@pytest.mark.gpu
def test_long_blend_chain_uploads(rt):
    """100 000 Blends in a row: the upload's check is iterative, so a deep graph costs no host recursion."""
    n = 100_000
    g = Graph()
    g.add(EMISSIVE, rgb=(1, 1, 1))
    for k in range(1, n):
        g.add(BLEND, k - 1, 0, scalar=0.5)
    sc = set_materials(rt, _two_spheres(rt), g.nodes, [n - 1, 0])
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
    finally:
        ctx.close()


def random_graph(rng):
    n = int(rng.integers(1, 13))
    nodes = []
    for _ in range(n):
        t = int(rng.choice((DIFFUSE, CHECKER, REFLECTIVE, EMISSIVE, NULL, BLEND, BLEND, COMBINE, COMBINE, COMBINE)))
        a, b = (int(x) for x in rng.integers(0, n, 2)) if t in (BLEND, COMBINE) else (-1, -1)
        scalar = {BLEND: rng.random(), CHECKER: rng.choice((0.2, 1.0, -0.5))}.get(t, 0.0)
        nodes.append((t, a, b, tuple(float(x) for x in rng.choice(LEVELS, 3)), float(scalar)))
    if rng.random() < 0.3:                              # long Combine chains, sometimes one too long
        base = len(nodes)
        depth = int(rng.integers(MAX_COMBINES - 1, MAX_COMBINES + 2))
        nodes.append((EMISSIVE, -1, -1, (0.25, 0.5, 0.25), 0.0))
        for k in range(depth):
            nodes.append((COMBINE, base + k, int(rng.integers(0, base + k + 1)), (0, 0, 0), 0.0))
    n = len(nodes)
    return nodes, [int(x) for x in rng.integers(-2 if rng.random() < 0.1 else -1, n, 2)]


@pytest.mark.gpu
def test_random_graphs_are_refused_exactly_by_the_rule(rt, restatement):
    """200 small graphs of random types and child indices (cycles are common): the upload accepts exactly the graphs
    upload_allowed accepts, and some accepted ones render as the restatement renders them."""
    rng = np.random.default_rng(2024)
    rays = random_rays(2000, 37)
    ctx = rt.GpuContext(0)
    try:
        verdicts, rendered = [], 0
        for k in range(200):
            nodes, roots = random_graph(rng)
            sc = set_materials(rt, _two_spheres(rt), nodes, roots)
            allowed = upload_allowed(nodes, roots)
            try:
                ctx.upload_scene(sc)
                accepted = True
            except rt.RtError:
                accepted = False
            assert accepted == allowed, (k, nodes, roots)
            verdicts.append(allowed)
            if accepted and rendered < 12 and any(nd[0] == COMBINE for nd in nodes):
                rendered += 1
                for mode in (PATH, PREVIEW):
                    want, _ = restatement.radiance_rays(sc.desc, rays, mode, 6, k, 0, np.arange(len(rays)), 0)
                    assert same_bits(radiance(ctx, rays, mode=mode, max_bounce=6, seed=k)[:, :3], want), (k, mode)
        assert 20 <= sum(verdicts) <= 180 and rendered >= 5, (sum(verdicts), rendered)
    finally:
        ctx.close()
