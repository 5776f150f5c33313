"""Generates the committed golden fixtures FROM THE REFERENCE ITSELF.

The reference ships no golden vectors (SURVEY.md §4), so these are outputs of its own unmodified code,
compiled in place by oracle/Makefile into oracle/_ref/libref_oracle.so and driven through
oracle/ref_harness.cpp with the shared counter RNG.  Run where /root/reference exists:

    python tests/golden/make_golden.py

Without the reference, `--standin` writes the fixtures of the generated stand-in meshes
(tests/standin_data.py) into tests/golden/standin/, at reduced sizes, through the plain-C restatement
in the reference's place (tests/port_reference.py; tests/test_oracle_vs_ref.py pins it to the
reference).  They pin the CUDA path and the host layer to what the restatement computed when they
were written.  kat.npz holds no mesh and is not rewritten.

Inputs are regenerated from fixed seeds by the tests; the fixtures hold inputs too where that is cheap,
so a change of numpy's generators cannot silently invalidate them.
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import scenes  # noqa: E402
from oracle.bindings import RefOracle  # noqa: E402
from test_gpu_parity import random_rays  # noqa: E402

DATA = os.path.join(ROOT, "assets", "_ref", "Data")

RENDERS = {
    # name: (scene, W, H, mode, max_bounce, antialias, passes, seed, table_seed)
    "c1_whitted": ("c1_torusknot", 160, 120, 2, 1, 0, 1, 0, None),
    "c2_reflective": ("c2_monkey", 160, 90, 0, 5, 0, 1, 0, None),
    "c2_null": ("c2_monkey_null", 160, 90, 0, 5, 0, 1, 0, None),
    "mix_deterministic": ("deterministic_mix", 160, 90, 0, 10, 0, 1, 0, None),
    "c3_preview": ("c3_unitychan", 160, 90, 1, 10, 1, 1, 3, None),
    "c3_path": ("c3_unitychan", 120, 68, 0, 10, 1, 4, 0, 0),
    "default_path": ("default_scene", 96, 96, 0, 10, 1, 2, 11, 5),
}


def main_standin():
    import raytracerwin_b200 as rt
    import standin_data
    from oracle.bindings import PortOracle
    from port_reference import PortReference
    rt.load_library()
    ref = PortReference(rt, PortOracle())
    with tempfile.TemporaryDirectory() as tmp:
        data = standin_data.write(os.path.join(tmp, "Data"))
        write_mesh_fixtures(ref, data, os.path.join(HERE, "standin"), scale=2, n_rays=2000, n_uv=500)


def main():
    ref = RefOracle()
    kat(ref)
    write_mesh_fixtures(ref, DATA, HERE)


def kat(ref):
    rng = np.random.default_rng(3)
    n = 4000
    rays = random_rays(n, 11)
    lo = rng.normal(size=(n, 3)).astype(np.float32)
    ext = np.abs(rng.normal(size=(n, 3))).astype(np.float32)
    ext[: n // 8, 0] = 0.0
    boxes = np.concatenate([lo, lo + ext], 1)
    tris = (rng.normal(size=(n, 9)) * 1.5).astype(np.float32)
    tris[: n // 10, 3:6] = tris[: n // 10, 0:3] + (rng.normal(size=(n // 10, 3)) * 1e-4).astype(np.float32)
    spheres = np.concatenate([rng.normal(size=(n, 3)), np.abs(rng.normal(size=(n, 1))) + 0.1], 1).astype(np.float32)
    planes = np.concatenate([rng.normal(size=(n, 3)), rng.normal(size=(n, 3))], 1).astype(np.float32)
    caps = np.concatenate([rng.normal(size=(n, 6)), np.abs(rng.normal(size=(n, 1))) * 0.5 + 0.05], 1).astype(np.float32)
    x = (np.abs(rng.normal(size=n)).astype(np.float32) * np.float32(10) ** rng.integers(-6, 6, n).astype(np.float32)).astype(np.float32)
    pabc = rng.normal(size=(n, 12)).astype(np.float32)
    rgb = (rng.random(size=(n, 3)) * 1.2).astype(np.float32)
    out = dict(rays=rays, boxes=boxes, tris=tris, spheres=spheres, planes=planes, caps=caps, x=x, pabc=pabc, rgb=rgb)
    out["aabb_hit"], out["aabb_tmin"] = ref.kat_aabb(rays, boxes)
    out["tri_hit"], out["tri_out"] = ref.kat_triangle(rays, tris)
    out["sphere_hit"], out["sphere_out"] = ref.kat_sphere(rays, spheres)
    out["plane_hit"], out["plane_out"] = ref.kat_plane(rays, planes)
    out["capsule_hit"], out["capsule_out"] = ref.kat_capsule(rays, caps)
    out["qrsqrt"] = ref.kat_qrsqrt(x)
    out["bary"] = ref.kat_barycentric(pabc)
    out["display"] = ref.kat_display(rgb)
    np.savez_compressed(os.path.join(HERE, "kat.npz"), **out)


def write_mesh_fixtures(ref, DATA, OUT, scale=1, n_rays=20000, n_uv=2000):
    """Fixtures of scenes with meshes from DATA into OUT; image sides divided by `scale`."""
    os.makedirs(OUT, exist_ok=True)
    # loader + BVH + primary hits per mesh
    for name in ("TorusKnot", "BlenderMonkey", "unitychan"):
        spec = [("mesh", f"{DATA}/{name}.obj", ("diffuse", scenes.WHITE))]
        s = ref.build_scene(spec)
        counts = np.array(ref.mesh_counts(s, 0), np.int32)
        bounds, escape, tri, verts = ref.mesh_bvh(s, 0)
        d = ref.mesh_dump(s, 0)
        W, H = 160 // scale, 120 // scale
        r = ref.trace_primary(s, W, H, want_hit=isinstance(ref, RefOracle))
        assert r["mismatches"] == 0
        digest = lambda a: np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)
        hit = {} if r["hit"] is None else dict(hit=r["hit"])
        np.savez_compressed(os.path.join(OUT, f"primary_{name}.npz"), counts=counts, W=W, H=H, **hit,
                            bvh_bounds_sha=digest(bounds), bvh_escape_sha=digest(escape), bvh_tri_sha=digest(tri),
                            points_sha=digest(d["points"]), pidx_sha=digest(d["pidx"]), matid_sha=digest(d["matid"]),
                            shape=r["shape"].astype(np.int8), tri=r["tri"], dist=r["dist"],
                            node_tests=r["node_tests"], tri_tests=r["tri_tests"])
        if name == "unitychan":
            # texture pixels (linearised by the reference at load): digest per slot + a few samples
            tex = {}
            uv = (np.random.default_rng(5).random(size=(n_uv, 2)) * 3 - 1).astype(np.float32)
            k = 0
            for slot in range(16):
                px = ref.mesh_texture(s, 0, slot)
                if px is None:
                    continue
                tex[f"tex{k}_slot"] = slot
                tex[f"tex{k}_shape"] = np.array(px.shape[:2], np.int32)
                tex[f"tex{k}_sha"] = digest(px)
                tex[f"tex{k}_samples"] = ref.kat_texture_sample(s, 0, slot, uv)
                k += 1
            np.savez_compressed(os.path.join(OUT, "textures_unitychan.npz"), uv=uv, count=k, **tex)
        ref.free_scene(s)

    # arbitrary rays through the default scene (all shape classes)
    s = ref.build_scene(scenes.default_scene(DATA))
    rr = random_rays(n_rays, 7)
    sh, tr, hit = ref.trace_rays(s, rr)
    np.savez_compressed(os.path.join(OUT, "rays_default_scene.npz"), rays=rr, shape=sh.astype(np.int8), tri=tr, hit=hit)
    ref.free_scene(s)

    # renders
    for name, (scene, W, H, mode, bounce, aa, passes, seed, table_seed) in RENDERS.items():
        W, H = W // scale, H // scale
        if table_seed is not None:
            ref.init_unit_vectors(table_seed)
        s = ref.build_scene(getattr(scenes, scene)(DATA))
        r = ref.render(s, W, H, mode=mode, max_bounce=bounce, antialias=aa, pass_count=passes, seed=seed, nthreads=8, want_display=True)
        np.savez_compressed(os.path.join(OUT, f"render_{name}.npz"), accum=r["accum"], display=r["display"],
                            params=np.array([W, H, mode, bounce, aa, passes, seed, -1 if table_seed is None else table_seed], np.int32))
        ref.free_scene(s)
        print(name, "done")
    total = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT) if f.endswith(".npz"))
    print("fixtures:", total // 1024, "KiB")


if __name__ == "__main__":
    main_standin() if "--standin" in sys.argv[1:] else main()
