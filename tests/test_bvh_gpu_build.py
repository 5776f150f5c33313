"""SURVEY 8f-1: KdTree::Build on the device == the host builder (itself pinned to the reference's tree by
tests/test_oracle_vs_ref.py), bit for bit: node bounds, escape links, leaf slots, triangle records, depth.

A numpy restatement of the build (`restate`) is a second reference that needs no compiled reference: the CPU tests
hold it to the host builder on adversarial meshes and prove, with it, that each generator reaches the edge it is
named for; the GPU tests hold the device builder and its three callers (rt_gpu_build_bvh, the loader's device
builder, rt_gpu_update_mesh / rt_gpu_replace_mesh) to the host builder on the same meshes and at the sizes where the
device's scans carry across chunks."""
import os
import sys
import types

import numpy as np
import pytest

from conftest import ROOT
from test_scene_replace import ReplaceExpected, replace
from test_scene_updates import Expected, check_arrays, check_results, deform, fresh, make_scene, update

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_c5  # noqa: E402

F32 = np.float32
FMAX = np.finfo(F32).max
TINY = np.finfo(F32).tiny                   # smallest normal float32
NODE_DT = np.dtype([("bmin", "<f4", 3), ("escape", "<i4"), ("bmax", "<f4", 3), ("tri", "<i4")])
BIG_SEG, SUM_TILE, WARP, BLOCK = 512, 1024, 32, 256     # rt_bvh_build.cu: serial-sum threshold and tile, k_bounds launch
SCAN_CHUNK = 1024 * 1024                    # k_scan_sums carries a running total past this many triangles


# ---------------------------------------------------------------------------------------------------
# the restatement of KdNode::Build (KdTree.cpp:10-126), in the rules of rt_bvh_build.cu's header
# ---------------------------------------------------------------------------------------------------
def seq_sum(v):
    """fp32 sum in list order, one rounding per addition (np.sum would sum pairwise)."""
    return np.add.accumulate(v, dtype=F32)[-1]


def restate(points, pidx):
    """The tree as Scene.flat_mesh emits it: nodes (pre-order, NODE_DT), the triangle id of each leaf slot, the
    depth, and per split node a record (begin, ids in list order, axis, mean, left count before the fallback)."""
    P = np.ascontiguousarray(points, F32).reshape(-1, 3)
    I = np.ascontiguousarray(pidx, np.int32).reshape(-1, 3)
    T = len(I)
    V = P[I]                                                     # (T, corner, axis)
    with np.errstate(over="ignore"):
        C = ((V[:, 0] + V[:, 1]) + V[:, 2]) / F32(3)            # (v0 + v1 + v2) / 3, left to right
    nodes = np.zeros(2 * T - 1, NODE_DT)
    order = np.arange(T)
    splits, depth = [], 0
    stack = [(0, T, 0, 1)]                                       # begin, end, node, level
    while stack:
        b, e, node, level = stack.pop()
        depth = max(depth, level)
        n, ids = e - b, order[b:e].copy()
        corners = V[ids].reshape(-1, 3)                          # list order: triangle by triangle, corner by corner
        # the first corner that attains the extreme supplies the bits; == treats -0 and +0 as equal
        lo = np.array([corners[np.flatnonzero(corners[:, c] == corners[:, c].min())[0], c] for c in range(3)], F32)
        hi = np.array([corners[np.flatnonzero(corners[:, c] == corners[:, c].max())[0], c] for c in range(3)], F32)
        nodes[node] = (lo, node + 2 * n - 1, hi, b if n == 1 else -1)
        if n == 1:
            continue
        with np.errstate(over="ignore"):
            ex, ey, ez = hi - lo
        axis = (0 if ex > ez else 2) if ex > ey else (1 if ey > ez else 2)
        v = C[ids, axis]
        with np.errstate(over="ignore", invalid="ignore"):
            mean = seq_sum(v) / F32(n)
            left = v < mean                                      # strict, so NaN sends everything right
        nl = int(left.sum())
        if 0 < nl < n:
            order[b:e] = np.concatenate([ids[left], ids[~left]])     # stable
            mid = nl
        else:
            mid = n // 2                                         # all on one side: first half / second half
        splits.append(types.SimpleNamespace(begin=b, node=node, ids=ids, axis=axis, mean=mean, nl=nl, v=v))
        stack.append((b + mid, e, node + 2 * mid, level + 1))
        stack.append((b, b + mid, node + 1, level + 1))
    return types.SimpleNamespace(nodes=nodes, order=order, depth=depth, splits=splits, V=V, C=C)


def host_scene(rt, points, pidx):
    sc = rt.Scene()
    sc.add_mesh_arrays(points, pidx, material=("diffuse", (1, 1, 1)))
    return sc


# ---------------------------------------------------------------------------------------------------
# adversarial meshes: seeded, float32, each proven to reach its edge by the restatement (tests below)
# ---------------------------------------------------------------------------------------------------
def loose(rng, pts):
    """One triangle per three points, in a shuffled order."""
    pts = np.asarray(pts, F32).reshape(-1, 3)
    perm = rng.permutation(len(pts) // 3)
    return pts, (3 * perm[:, None] + np.arange(3)).astype(np.int32)


def signed_zeros(seed=1, T=3000):
    """x >= 0 and z <= 0 everywhere, with the extreme 0 reached by corners of both signs at random list positions:
    ties of -0 and +0 within and across warps and blocks of k_bounds."""
    rng = np.random.default_rng(seed)
    P = 3 * T // 2
    pts = np.stack([rng.uniform(0.05, 1, P), rng.uniform(-0.6, 0.6, P), rng.uniform(-1, -0.05, P)], 1).astype(F32)
    for c in (0, 2):
        z = rng.random(P) < 0.04
        pts[z, c] = np.where(rng.random(z.sum()) < 0.5, F32(-0.0), F32(0.0))
    return pts, rng.integers(0, P, (T, 3)).astype(np.int32)


def mean_ties(seed=2, m=120):
    """Centroids exactly equal to their node's mean: m triangles at each integer x in [-3, 3] (sums exact), and a
    cluster at x = 1024 whose centroids sit one ulp below, at and one ulp above its mean of 1024."""
    rng = np.random.default_rng(seed)
    xs = np.repeat(np.arange(-3, 4), m).astype(F32)
    yz = rng.uniform(0, 0.4, (len(xs), 3, 2)).astype(F32)
    a = np.concatenate([np.broadcast_to(xs[:, None, None], (len(xs), 3, 1)), yz], 2)
    near = np.repeat(np.array([np.nextafter(F32(1024), F32(0)), F32(1024), np.nextafter(F32(1024), F32(2048))], F32), 20)
    b = np.zeros((len(near), 3, 3), F32)
    b[:, :, 0] = near[:, None]
    return loose(rng, np.concatenate([a, b]))


def order_sensitive(seed=3, sizes=(512, 513, 1024, 1025, 2049)):
    """Clusters of the given triangle counts at x ~ 1e7 (ulp 1), far apart on x so that each is a node: integer
    jitter of +-60 on x and +-20 on y, z.  Within a cluster the fp32 sum of ~1e10 rounds at every step, so another
    summation order moves the mean across centroids."""
    rng = np.random.default_rng(seed)
    out = []
    for k, n in enumerate(sizes):
        c = np.array([1.0e7 + 1.5e6 * k, 0, 0])
        out.append(c + np.concatenate([rng.integers(-60, 61, (n, 3, 1)), rng.integers(-20, 21, (n, 3, 2))], 2))
    return loose(rng, np.concatenate(out))


def same_centroid(seed=4, T=1025):
    """Every centroid identical: corners r, -r and one shared point K, so (r + -r) + K is K for every triangle.
    The half-split fallback runs at every level; the bounds still differ from node to node."""
    rng = np.random.default_rng(seed)
    r = rng.uniform(-2, 2, (T, 3)).astype(F32)
    pts = np.concatenate([np.array([[0.7, 0.2, -0.5]], F32), r, -r])
    pidx = np.stack([1 + np.arange(T), 1 + T + np.arange(T), np.zeros(T, int)], 1).astype(np.int32)
    return pts, pidx


def overflow(seed=5, T=1500):
    """Finite corners whose sums overflow: centroids of +inf and -inf (a NaN mean where both meet in a node), and
    nodes whose extent is inf on two and on three axes, among ordinary triangles."""
    rng = np.random.default_rng(seed)
    big = F32(0.75) * FMAX
    fam = rng.integers(0, 6, T)
    tri = rng.uniform(-1, 1, (T, 3, 3)).astype(F32)
    sgn = np.where(rng.random(T) < 0.5, F32(-1), F32(1))
    tri[fam == 1, :, 0] = (sgn[fam == 1] * big)[:, None]                         # centroid x = +-inf
    tri[fam == 2, :, 2] = (sgn[fam == 2] * big)[:, None]                         # centroid z = +-inf
    two = fam == 3                                                               # +-FLT_MAX on x and y: extents inf
    tri[two, 0, :2], tri[two, 1, :2] = FMAX, -FMAX
    three = fam == 4                                                             # ... and on z
    tri[three, 0], tri[three, 1] = FMAX, -FMAX
    return loose(rng, tri)


def denormals(seed=6, T=1200):
    """Every corner, centroid and extent below the smallest normal float32: multiples of 2^-149 up to 3000 of them
    (x) and 800 (y, z).  A flush to zero would send every triangle to one side."""
    rng = np.random.default_rng(seed)
    q = np.concatenate([rng.integers(-3000, 3001, (T, 3, 1)), rng.integers(-800, 801, (T, 3, 2))], 2)
    return loose(rng, q.astype(F32) * F32(2.0 ** -149))


def geometric(seed=7, T=1200):
    """Deep, unbalanced trees: triangles of corners (x, 0, 0), the origin and the origin, with |x| spaced geometrically
    over the float range and random signs, so that each split peels off the few triangles of largest magnitude."""
    rng = np.random.default_rng(seed)
    x = (np.geomspace(1e-44, 1e38, T) * np.where(rng.random(T) < 0.5, -1, 1)).astype(F32)
    pts = np.zeros((T + 1, 3), F32)
    pts[1:, 0] = x
    pidx = np.stack([1 + rng.permutation(T), np.zeros(T, int), np.zeros(T, int)], 1).astype(np.int32)
    return pts, pidx


def shared_points(seed=8, P=400, T=900):
    """Repeated index triples, the same corners in other orders, triangles on one or two points, and points no
    triangle uses (placed outside the used ones, so they would widen any bound they reached)."""
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-1, 1, (P, 3)).astype(F32)
    pts[-40:] = rng.uniform(5, 1e30, (40, 3)).astype(F32) * np.where(rng.random((40, 3)) < 0.5, -1, 1).astype(F32)
    base = rng.integers(0, P - 40, (T // 3, 3))
    rep = base[rng.integers(0, len(base), T // 3)]                                 # exact repeats
    rot = base[rng.integers(0, len(base), T - 2 * (T // 3))][:, [1, 2, 0]]          # same corners, another order
    pidx = np.concatenate([base, rep, rot])
    pidx[::17] = pidx[::17, :1]                                                    # one point three times
    pidx[5::19, 1] = pidx[5::19, 0]                                                # two points
    return pts, pidx[rng.permutation(T)].astype(np.int32)


GENERATORS = {
    "signed_zeros": signed_zeros,
    "mean_ties": mean_ties,
    "order_sensitive": order_sensitive,
    "same_centroid_1025": lambda: same_centroid(T=1025),
    "same_centroid_4097": lambda: same_centroid(T=4097),
    "overflow": overflow,
    "denormals": denormals,
    "geometric": geometric,
    "shared_points": shared_points,
}


# ---------------------------------------------------------------------------------------------------
# 1. the restatement equals the host builder (no GPU)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(GENERATORS))
def test_restatement_equals_host_build(rt, name):
    pts, pidx = GENERATORS[name]()
    r = restate(pts, pidx)
    sc = host_scene(rt, pts, pidx)
    nodes, tris, _ = sc.flat_mesh(0)
    assert nodes.tobytes() == r.nodes.tobytes()
    np.testing.assert_array_equal(tris["index"], r.order)
    for k in range(3):
        assert tris[f"p{k}"].tobytes() == r.V[r.order, k].tobytes()
    assert sc.mesh_counts(0)[6] == r.depth


# ---------------------------------------------------------------------------------------------------
# 2. each generator reaches its edge (no GPU)
# ---------------------------------------------------------------------------------------------------
def zero_ties(r, c, side):
    """Per split node whose bound `side` ("min" | "max") on axis c is 0: the tying corners' list positions and signs."""
    out = []
    for s in r.splits:
        col = r.V[s.ids, :, c].ravel()
        if (col.min() if side == "min" else col.max()) == 0:
            k = np.flatnonzero(col == 0)
            out.append((s.begin + k // 3, np.signbit(col[k])))
    return out


def test_signed_zeros_reach_warp_and_block_ties():
    r = restate(*signed_zeros())
    for c, side in ((0, "min"), (2, "max")):
        ties = zero_ties(r, c, side)
        for first in (True, False):                 # -0 first, then +0 first
            mine = [(p, s) for p, s in ties if s[0] == first]
            # an opposite-signed tie in another block of k_bounds, and one in another warp of the same block
            assert any(((p // BLOCK != p[0] // BLOCK) & (s != first)).any() for p, s in mine), (c, first)
            assert any(((p // BLOCK == p[0] // BLOCK) & (p // WARP != p[0] // WARP) & (s != first)).any() for p, s in mine), (c, first)
            # the last tie has the other sign: keeping the last corner instead of the first changes the bits
            assert any(s[-1] != first and p[-1] // BLOCK != p[0] // BLOCK for p, s in mine), (c, first)


def test_mean_ties_reach_equality_and_ulps():
    r = restate(*mean_ties())
    equal = [s for s in r.splits if (s.v == s.mean).any()]
    assert any((s.v <= s.mean).sum() != s.nl for s in equal)
    assert len(equal) >= 3
    assert any((s.v == np.nextafter(s.mean, F32(-np.inf))).any() and (s.v == np.nextafter(s.mean, F32(np.inf))).any()
               and (s.v == s.mean).any() for s in r.splits)


def pairwise_sum(v):
    return v[0] if len(v) == 1 else pairwise_sum(v[:len(v) // 2]) + pairwise_sum(v[len(v) // 2:])


def tiles_reversed(v):
    return np.concatenate([v[k:k + SUM_TILE] for k in range(0, len(v), SUM_TILE)][::-1])


def test_order_sensitive_means_move_partitions():
    r = restate(*order_sensitive())
    counts = {len(s.ids) for s in r.splits}
    assert {512, 513, 1024, 1025, 2049} <= counts

    def nl(s, total):
        return int((s.v < total / F32(len(s.v))).sum())

    big = [s for s in r.splits if len(s.ids) > BIG_SEG]
    assert any(nl(s, pairwise_sum(s.v)) != s.nl for s in big)
    assert any(nl(s, seq_sum(s.v[::-1])) != s.nl for s in big)
    # k_sum_big's tiles added in another order: a different split in a node of more than one tile
    assert any(nl(s, seq_sum(tiles_reversed(s.v))) != s.nl for s in big if len(s.ids) > SUM_TILE)
    assert all(nl(s, seq_sum(s.v)) == s.nl for s in r.splits)


@pytest.mark.parametrize("T", [1025, 4097])
def test_same_centroid_falls_back_at_every_level(T):
    pts, pidx = same_centroid(T=T)
    r = restate(pts, pidx)
    assert (r.C == r.C[0]).all()
    assert len(r.splits) == T - 1 and all(s.nl in (0, len(s.ids)) for s in r.splits)
    assert len({r.nodes[s.node]["bmin"].tobytes() for s in r.splits}) > T // 2


def test_overflow_reaches_inf_centroids_nan_means_and_inf_extents():
    pts, pidx = overflow()
    assert np.isfinite(pts).all()
    r = restate(pts, pidx)
    assert np.isposinf(r.C).any() and np.isneginf(r.C).any()
    nan = [s for s in r.splits if np.isnan(s.mean)]
    assert nan and all(s.nl == 0 for s in nan)
    assert any(np.isposinf(s.v).any() and np.isneginf(s.v).any() for s in nan)
    assert any(np.isinf(s.mean) for s in r.splits)
    with np.errstate(over="ignore"):
        inf_axes = [int(np.isinf(r.nodes[s.node]["bmax"] - r.nodes[s.node]["bmin"]).sum()) for s in r.splits]
    assert {1, 2, 3} <= set(inf_axes)
    # two infinite extents pick y (x is not strictly wider), three pick z
    assert any(n == 2 and s.axis == 1 for n, s in zip(inf_axes, r.splits))
    assert any(n == 3 and s.axis == 2 for n, s in zip(inf_axes, r.splits))


def test_denormals_split_where_a_flush_would_not():
    pts, pidx = denormals()
    assert (np.abs(pts) < TINY).all() and (pts != 0).any()
    r = restate(pts, pidx)
    assert (np.abs(r.C) < TINY).all()

    def ftz(x):
        return np.where(np.abs(x) < TINY, F32(0), x)

    assert any((ftz(s.v) < ftz(s.mean)).sum() != s.nl for s in r.splits)
    assert any(((r.nodes[s.node]["bmax"] != 0) & (np.abs(r.nodes[s.node]["bmax"]) < TINY)).any() for s in r.splits)


def test_geometric_centroids_make_a_deep_tree():
    pts, pidx = geometric()
    r = restate(pts, pidx)
    assert r.depth >= 75 > 6 * np.log2(len(pidx))             # 79 for this seed; a balanced tree has 12 levels
    assert np.isfinite(r.C).all() and (np.abs(r.C[r.C != 0]) < TINY).any() and (np.abs(r.C) > 1e37).any()


def test_shared_points_reach_repeats_and_unused_points():
    pts, pidx = shared_points()
    r = restate(pts, pidx)
    assert len(np.unique(pidx, axis=0)) < len(pidx)                            # repeated triples
    srt = np.sort(pidx, 1)
    same = (srt[:, None] == srt[None]).all(2) & ~(pidx[:, None] == pidx[None]).all(2)
    assert same.any()                                                           # same corners, another order
    assert (pidx[:, 0] == pidx[:, 2]).any() and ((pidx[:, 0] == pidx[:, 1]) & (pidx[:, 1] != pidx[:, 2])).any()
    far = np.arange(len(pts) - 40, len(pts))
    assert np.isin(far, np.setdiff1d(np.arange(len(pts)), pidx)).all()
    root = r.nodes[0]
    assert (((pts[far] < root["bmin"]) | (pts[far] > root["bmax"])).any(1)).all()


# ---------------------------------------------------------------------------------------------------
# 3. the device builder (GPU)
# ---------------------------------------------------------------------------------------------------
def check(rt, gpu, sc):
    d = sc.mesh_dump(0)
    nodes, tris, shade = sc.flat_mesh(0)
    gn, gt, depth, ms = gpu.build_bvh(d["points"], d["pidx"])
    assert depth == sc.mesh_counts(0)[6]
    assert gn.tobytes() == nodes.tobytes()
    assert gt.tobytes() == tris.tobytes()
    return ms


def jittered_grid(T, seed=0, mixed=False):
    """T triangles of a jittered height field over [-2, 2]^2 (the first T of a grid).  mixed: a column of x = +-0 and
    a row of y = +-0 corners, and patches of corners at +-0.75 FLT_MAX on z and on x (centroids of +-inf, NaN means,
    infinite extents)."""
    rng = np.random.default_rng(seed)
    n = max(1, int(np.ceil(np.sqrt(T / 2))))
    u = np.linspace(-2, 2, n + 1)
    X, Y = np.meshgrid(u, u)
    pts = np.stack([X, Y, 0.3 * np.sin(3 * X) * np.cos(2 * Y)], -1).reshape(-1, 3)
    pts = (pts + rng.uniform(-0.3, 0.3, pts.shape) * (4 / n)).astype(F32)
    a = (np.arange(n)[:, None] * (n + 1) + np.arange(n)[None, :]).ravel()
    pidx = np.stack([np.stack([a, a + 1, a + n + 2], 1), np.stack([a, a + n + 2, a + n + 1], 1)], 1).reshape(-1, 3)[:T]
    if mixed:
        P = pts.reshape(n + 1, n + 1, 3)
        sign = lambda shape: np.where(rng.random(shape) < 0.5, F32(-0.0), F32(0.0))
        P[:, n // 2, 0] = sign(n + 1)
        P[n // 3, :, 1] = sign(n + 1)
        big = F32(0.75) * FMAX
        for k in range(8):
            i, j = rng.integers(0, n - 3, 2)
            P[i:i + 4, j:j + 4, 2 if k < 6 else 0] = big if k % 2 else -big
    return pts, pidx.astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["TorusKnot", "BlenderMonkey", "unitychan"])
def test_gpu_build_equals_host_build(rt, gpu, data_dir, name):
    sc = rt.Scene([("mesh", f"{data_dir}/{name}.obj", ("diffuse", (1, 1, 1)))])
    check(rt, gpu, sc)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GENERATORS))
def test_gpu_build_adversarial_meshes(rt, gpu, name):
    check(rt, gpu, host_scene(rt, *GENERATORS[name]()))


@pytest.mark.gpu
@pytest.mark.parametrize("T,mixed", [(T, False) for T in (1, 2, 31, 32, 33, 511, 512, 513, 1023, 1024, 1025, 2049)]
                         + [(SCAN_CHUNK, False), (SCAN_CHUNK + 1, True), (3 * SCAN_CHUNK + 1, False)])
def test_gpu_build_sizes_at_chunk_edges(rt, gpu, T, mixed):
    """Block, warp and tile edges of the device kernels, and the scan of block sums with one, two and four chunks."""
    pts, pidx = jittered_grid(T, seed=T, mixed=mixed)
    assert len(pidx) == T
    check(rt, gpu, host_scene(rt, pts, pidx))


@pytest.mark.gpu
def test_gpu_build_generated_grid_and_degenerates(tmp_path, rt, gpu, data_dir):
    out = str(tmp_path / "torus_200.obj")
    make_c5.main(os.path.join(data_dir, "TorusKnot.obj"), out, 200)           # 240 k triangles, "-0.000000" coordinates included
    sc = rt.Scene([("mesh", out, ("diffuse", (1, 1, 1)))])
    ms = check(rt, gpu, sc)
    assert ms > 0
    # coincident centroids (half-split fallback), zero-area and repeated triangles, signed zeros
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [-0.0, 0.0, -0.0], [0.0, -0.0, 0.0], [2, 2, 2], [2, 2, 2], [2, 2, 2],
                    [1, 1, -0.0], [-1, 0.0, 0.0], [0.0, -1, 0.0]], np.float32)
    idx = np.array([[0, 1, 2], [0, 1, 2], [0, 1, 2], [3, 4, 3], [5, 6, 7], [0, 1, 2], [8, 9, 10], [3, 1, 2], [4, 1, 2], [0, 1, 2]], np.int32)
    sc2 = rt.Scene()
    sc2.add_mesh_arrays(pts, idx, material=("diffuse", (1, 1, 1)))
    check(rt, gpu, sc2)
    sc3 = rt.Scene()
    sc3.add_mesh_arrays(pts, idx[:1], material=("diffuse", (1, 1, 1)))      # a single triangle: the root is a leaf
    check(rt, gpu, sc3)


def device_built(rt, gpu, spec):
    rt.use_device_bvh_builder(gpu)
    try:
        return rt.Scene(spec)
    finally:
        rt.use_device_bvh_builder(None)


@pytest.mark.gpu
def test_scene_loader_with_device_builder(rt, gpu, port, data_dir):
    """The host scene layer with the device builder switched on: same flattened mesh, same render."""
    spec = [("mesh", f"{data_dir}/unitychan.obj", ("reflective", (0.8, 0.8, 0.8), 0.0))]
    host = rt.Scene(spec)
    dev = device_built(rt, gpu, spec)
    for a, b in zip(host.flat_mesh(0), dev.flat_mesh(0)):
        assert a.tobytes() == b.tobytes()
    assert host.mesh_counts(0) == dev.mesh_counts(0)
    gpu.upload_scene(dev)
    W, H = 320, 180
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=4, antialias=0)
    gpu.reset_accum(W, H)
    gpu.render_tile(p)
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    o = port.render(host.desc, p, nthreads=8)
    assert acc.tobytes() == o["accum"].tobytes()


@pytest.mark.gpu
def test_scene_loader_with_device_builder_past_scan_chunk(tmp_path, rt, gpu, data_dir):
    """A TorusKnot grid of more than 2^20 triangles through the loader's device builder equals the host-built scene."""
    src = os.path.join(data_dir, "TorusKnot.obj")
    T0 = rt.Scene([("mesh", src, None)]).mesh_counts(0)[3]
    copies = SCAN_CHUNK // T0 + 1
    out = str(tmp_path / "torus_grid.obj")
    make_c5.main(src, out, copies)
    spec = [("mesh", out, ("diffuse", (1, 1, 1)))]
    host = rt.Scene(spec)
    assert host.mesh_counts(0)[3] == copies * T0 > SCAN_CHUNK
    dev = device_built(rt, gpu, spec)
    for a, b in zip(host.flat_mesh(0), dev.flat_mesh(0)):
        assert a.tobytes() == b.tobytes()
    assert host.mesh_counts(0) == dev.mesh_counts(0)


@pytest.mark.gpu
def test_update_mesh_past_scan_chunk(rt):
    """rt_gpu_update_mesh rebuilds a tree of 2^20 + 1 triangles: the host build's arrays, and a fresh upload's results."""
    pts, pidx = jittered_grid(SCAN_CHUNK + 1, seed=11)
    sc = make_scene(rt, [("mesh_arrays", pts, pidx, ("diffuse", (0.8, 0.7, 0.6)))])
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        new = deform(pts, "wobble")
        update(ctx, 0, new, pidx)
        exp = Expected(rt, sc, 0, new)
        check_arrays(ctx, exp)
        ref = fresh(rt, exp.desc)
        try:
            check_results(rt, ctx, ref, modes=(0,))
        finally:
            ref.close()
    finally:
        ctx.close()


@pytest.mark.gpu
def test_update_mesh_with_overflowing_normals(rt):
    """Finite corners whose face normals overflow to NaN: the edit path's leaf and shading records carry the host
    build's bits."""
    pts, pidx = overflow()
    sc = make_scene(rt, [("mesh_arrays", pts, pidx, ("diffuse", (0.8, 0.7, 0.6)))])
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        new = deform(pts, "degenerate")
        exp = Expected(rt, sc, 0, new)
        assert np.isnan(exp.tris["n"]).any() and np.isnan(exp.shade["n0"]).any()
        update(ctx, 0, new, pidx)
        check_arrays(ctx, exp)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_replace_mesh_across_scan_chunk(rt):
    """rt_gpu_replace_mesh from 1 k triangles to 2^20 + 1 and back to 1 k (another mesh, into the grown scratch)."""
    pts, pidx = jittered_grid(1000, seed=12)
    sc = make_scene(rt, [("mesh_arrays", pts, pidx, ("diffuse", (0.8, 0.7, 0.6)))])
    ctx = rt.GpuContext(0)
    try:
        ctx.upload_scene(sc)
        for T, seed in ((SCAN_CHUNK + 1, 13), (1000, 14)):
            pts, pidx = jittered_grid(T, seed=seed)
            g = dict(points=pts, pidx=pidx)
            replace(ctx, 0, g)
            check_arrays(ctx, ReplaceExpected(rt, sc, 0, g))
    finally:
        ctx.close()
