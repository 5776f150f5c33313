"""Every BASELINE.json config AT ITS CONFIG SIZE against the unmodified reference (oracle/_ref/libref_oracle.so),
through the C-ABI — north_star: "bit-exact primary hits on every config".

  C4   unitychan 3840x2160: primary (shape, triangle) ids + Distance bits, exact and culled walks, and one full
       pass (4 jittered camera rays / pixel, MaxBounceTimes 10) of the accumulation buffer, bit for bit.
  C5s  62 translated copies (1.0 M triangles) 1920x1080: ids / Distance on a band of rows, one path pass on a band.
  C5   623 copies (10.0 M triangles) 3840x2160: the reference loads and builds the scene ONCE (about 80 s), its
       KdTree is compared node for node with the flattened array this repo uploads, then primary ids / Distance
       bits / node-test counts on bands of rows, and culled == exact on the whole 4K frame.

C1-C3 at their sizes are in test_gpu_parity.py.  The reference side reads only the staged assets and the
generated OBJ under RT_SCRATCH (default: a temporary directory of the test session).
Without the reference, the meshes are the generated stand-ins and the restatement takes the reference's
place (conftest.py).
"""
import os
import sys

import numpy as np
import pytest

import scenes
from conftest import DATA_DIR, ROOT, bits, is_reference, same_bits

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_c5  # noqa: E402

pytestmark = pytest.mark.gpu

WHITE = (1.0, 1.0, 1.0)
CORES = os.cpu_count() or 1


def primary(rt, gpu, W, H, traverse, start=0, end=None):
    end = W * H - 1 if end is None else end
    gpu.reset_accum(W, H)
    gpu.reset_counters()
    gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=traverse, start=start, end=end))
    ids = gpu.readback(rt.RT_READ_PRIMARY_IDS_I32X2, W, H).reshape(-1, 2)[start:end + 1]
    dist = gpu.readback(rt.RT_READ_PRIMARY_DIST_F32, W, H).reshape(-1)[start:end + 1]
    return ids, dist, gpu.counters()


def check_primary(rt, gpu, ref, rs, W, H, start=0, end=None, min_hits=1000):
    r = ref.trace_primary(rs, W, H, start=start, end=end)
    assert r["mismatches"] == 0
    assert (r["shape"] >= 0).sum() >= min_hits
    for tr in (rt.RT_TRAVERSE_EXACT, rt.RT_TRAVERSE_CULLED):
        ids, dist, c = primary(rt, gpu, W, H, tr, start, end if end is not None else W * H - 1)
        np.testing.assert_array_equal(ids[:, 0], r["shape"])
        np.testing.assert_array_equal(ids[:, 1], r["tri"])
        np.testing.assert_array_equal(bits(dist), bits(r["dist"]))
        if tr == rt.RT_TRAVERSE_EXACT:
            # the device walks exactly the nodes and triangles the reference walks
            assert c["node_tests"] == r["node_tests"] and c["tri_tests"] == r["tri_tests"]
        else:
            assert c["node_visits"] <= r["node_tests"] and c["tri_visits"] <= r["tri_tests"]
    return r


@pytest.fixture(scope="session")
def c5_dir(tmp_path_factory):
    """Where generated OBJs go: RT_SCRATCH (kept between runs) or a directory of this session."""
    out_dir = os.environ.get("RT_SCRATCH") or str(tmp_path_factory.mktemp("c5"))
    os.makedirs(out_dir, exist_ok=True)
    return out_dir


def generated(out_dir, data_dir, copies, aspect):
    src = os.path.join(data_dir, "unitychan.obj")
    out = os.path.join(out_dir, make_c5.cached_name(src, copies, aspect))
    if not os.path.exists(out):
        make_c5.main(src, out, copies, aspect)
    return [("mesh", out, ("blend", ("reflective", WHITE, 0.2), ("diffuse", WHITE), 1.0))]


def unitychan_triangles(rt, data_dir):
    """Triangles of one copy: 16056 in the reference's unitychan.obj."""
    n = rt.Scene([("mesh", os.path.join(data_dir, "unitychan.obj"), ("diffuse", WHITE))]).mesh_counts(0)[3]
    if data_dir == DATA_DIR:
        assert n == 16056
    return n


# ---------------------------------------------------------------------------------------------------
# C4: unitychan 3840x2160
# ---------------------------------------------------------------------------------------------------
def test_c4_primary_ids_and_one_pass_vs_reference(rt, gpu, ref, ref_counting, data_dir):
    spec = scenes.c3_unitychan(data_dir)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=0, count=0)
    gpu.upload_scene(sc)
    W, H = 3840, 2160
    rs = ref.build_scene(spec)
    check_primary(rt, gpu, ref, rs, W, H, min_hits=100_000)
    ref.free_scene(rs)
    # the passes go through the counting twin: its "rays" is the number of FindIntersectionWithScene calls
    ref = ref_counting
    ref.init_unit_vectors(0)
    rs = ref.build_scene(spec)
    # one full pass of the BASELINE frame: 4 jittered camera rays per pixel, MaxBounceTimes 10, seed 0
    r = ref.render(rs, W, H, mode=0, max_bounce=10, pass_begin=0, pass_count=1, antialias=1, seed=0, nthreads=CORES)
    gpu.reset_accum(W, H)
    gpu.reset_counters()
    gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, pass_begin=0, pass_count=1, antialias=1, seed=0))
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert np.abs(acc[..., :3] - r["accum"][..., :3]).max() <= 1e-4          # the bar north_star states ...
    assert np.array_equal(bits(acc), bits(r["accum"]))                        # ... and what actually holds
    assert gpu.counters()["rays"] == r["rays"]
    # a later pass of the same frame (other RNG keys), accumulated on top by both sides
    r2 = ref.render(rs, W, H, mode=0, max_bounce=10, pass_begin=9, pass_count=1, antialias=1, seed=0, nthreads=CORES,
                    accum=r["accum"])
    gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, pass_begin=9, pass_count=1, antialias=1, seed=0))
    assert np.array_equal(bits(gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)), bits(r2["accum"]))
    ref.free_scene(rs)


# ---------------------------------------------------------------------------------------------------
# C5s: 1.0 M triangles, 1920x1080
# ---------------------------------------------------------------------------------------------------
def test_c5s_band_vs_reference(rt, gpu, ref_counting, data_dir, c5_dir):
    ref = ref_counting
    W, H = 1920, 1080
    spec = generated(c5_dir, data_dir, 62, W / H)
    sc = rt.Scene(spec)
    sc.set_unit_vectors(seed=0, count=0)
    ref.init_unit_vectors(0)
    assert sc.mesh_counts(0)[3] == 62 * unitychan_triangles(rt, data_dir)
    gpu.upload_scene(sc)
    rs = ref.build_scene(spec)
    if is_reference(ref, "C5s loader counts"):
        assert sc.mesh_counts(0) == ref.mesh_counts(rs, 0)
    # primary hits: two bands of rows away from the centre row (whose rays have dy == 0: a disabled slab axis,
    # RRay.cpp:105, thousands of nodes each) and one across it
    hits = 0
    for row0, rows in ((H // 4, 48), (H // 2 - 4, 8), (3 * H // 4, 48)):
        r = check_primary(rt, gpu, ref, rs, W, H, start=row0 * W, end=(row0 + rows) * W - 1, min_hits=0)
        hits += int((r["shape"] >= 0).sum())
    assert hits >= 10_000
    # one path pass on a band through the figures
    start, end = (H // 2 - 16) * W, (H // 2 + 16) * W - 1
    r = ref.render(rs, W, H, mode=0, max_bounce=10, pass_begin=0, pass_count=1, antialias=1, seed=0, nthreads=CORES, start=start, end=end)
    gpu.reset_accum(W, H)
    gpu.reset_counters()
    gpu.render_tile(rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=10, pass_count=1, antialias=1, seed=0, start=start, end=end))
    acc = gpu.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H)
    assert same_bits(acc, r["accum"])
    assert gpu.counters()["rays"] == r["rays"]
    ref.free_scene(rs)


# ---------------------------------------------------------------------------------------------------
# C5: 10.0 M triangles, 3840x2160
# ---------------------------------------------------------------------------------------------------
def test_c5_ten_million_triangles_vs_reference(rt, gpu, ref, data_dir, c5_dir):
    W, H = 3840, 2160
    spec = generated(c5_dir, data_dir, 623, W / H)
    sc = rt.Scene(spec)
    per_copy = unitychan_triangles(rt, data_dir)
    assert sc.mesh_counts(0)[3] == 623 * per_copy
    gpu.upload_scene(sc)
    rs = ref.build_scene(spec)                          # the reference's loader + KdTree build: ~80 s
    nodes, tris, _ = sc.flat_mesh(0)
    assert len(nodes) == 2 * 623 * per_copy - 1
    if is_reference(ref, "C5 loader counts and tree node for node"):
        assert sc.mesh_counts(0) == ref.mesh_counts(rs, 0)
        # the tree, node for node (KdTree.cpp:37-126 against host/bvh_build.cpp)
        bounds, escape, tri, _ = ref.mesh_bvh(rs, 0)
        assert len(nodes) == len(escape)
        np.testing.assert_array_equal(nodes["escape"], escape)
        np.testing.assert_array_equal(bits(nodes["bmin"]), bits(bounds[:, :3]))
        np.testing.assert_array_equal(bits(nodes["bmax"]), bits(bounds[:, 3:]))
        leaf = nodes["tri"] >= 0
        np.testing.assert_array_equal(leaf, tri >= 0)
        np.testing.assert_array_equal(tris["index"][nodes["tri"][leaf]], tri[leaf])
        del bounds, escape, tri
    # primary hits on bands of rows (ids, Distance bits, node / triangle test counts)
    hits = 0
    for row0, rows in ((H // 4, 6), (H // 2 + 40, 6), (7 * H // 8, 6)):
        r = check_primary(rt, gpu, ref, rs, W, H, start=row0 * W, end=(row0 + rows) * W - 1, min_hits=0)
        hits += int((r["shape"] >= 0).sum())
    assert hits >= 5_000
    ref.free_scene(rs)
    # the whole frame: the culled walk finds what the exact walk finds
    e_ids, e_dist, ce = primary(rt, gpu, W, H, rt.RT_TRAVERSE_EXACT)
    c_ids, c_dist, cc = primary(rt, gpu, W, H, rt.RT_TRAVERSE_CULLED)
    np.testing.assert_array_equal(e_ids, c_ids)
    np.testing.assert_array_equal(bits(e_dist), bits(c_dist))
    assert (e_ids[:, 0] >= 0).mean() > 0.15
    assert cc["node_visits"] < ce["node_visits"]
