"""The reference's harness API (oracle.bindings.RefOracle), answered by the plain-C restatement
(oracle/librt_oracle.so) over the product's host scene layer.

The GPU tests compare the CUDA path with the unmodified reference where oracle/Makefile has built it
(oracle/_ref/).  Without it they compare with this instead: the restatement renders from the same
rt_scene_desc as the CUDA path, and tests/test_oracle_vs_ref.py pins it, bit for bit, to the reference
(loader, tree, textures, unit-vector table, primary hits, ray casts, every render mode, ray counts).
Its scenes, tree, textures and unit-vector table are the host layer's own, so they are no check of that
layer: tests leave those comparisons out when this stands in (conftest.is_reference).
tests/golden/make_golden.py --standin writes the fixtures of the stand-in meshes through it as well.
"""
import os
import time

import numpy as np

MODE_PATH, MODE_PREVIEW, MODE_WHITTED = 0, 1, 2


class PortReference:
    # its scenes, tree and unit-vector table are the host layer's own: conftest.is_reference() keeps tests from
    # comparing those with themselves
    stands_in = True

    def __init__(self, rt, port):
        self.rt, self.port, self.seed = rt, port, 0
        self._table = None

    # -- scenes: the product's host layer builds them (tests/test_oracle_vs_ref.py: as the reference does)
    def build_scene(self, shapes):
        s = self.rt.Scene(shapes)
        s._unit_seed = None
        return s

    def free_scene(self, s):
        pass

    def init_unit_vectors(self, seed=0):
        self.seed = seed

    def unit_vector_table(self):
        self._table = self.rt.Scene([])
        self._table.set_unit_vectors(seed=self.seed, count=0)
        d = self._table.desc.contents
        return np.ctypeslib.as_array(d.unit_vectors, (d.num_unit_vectors * 3,)).reshape(-1, 3)

    def _tables(self, s):
        # the reference's table is global state (init_unit_vectors); a host scene carries its own
        if s._unit_seed != self.seed:
            s.set_unit_vectors(seed=self.seed, count=0)
            s._unit_seed = self.seed

    def mesh_counts(self, s, shape):
        return s.mesh_counts(shape)

    def mesh_dump(self, s, shape):
        return s.mesh_dump(shape)

    def mesh_texture(self, s, shape, slot):
        return s.mesh_texture(shape, slot)

    def mesh_bvh(self, s, shape):
        nodes, tris, _ = s.flat_mesh(shape)
        bounds = np.concatenate([nodes["bmin"], nodes["bmax"]], 1)
        tri = np.where(nodes["tri"] >= 0, tris["index"][np.maximum(nodes["tri"], 0)], -1).astype(np.int32)
        return bounds, nodes["escape"], tri, np.zeros((len(tri), 3), np.int32)

    # -- tracing
    def trace_primary(self, s, W, H, start=0, end=None, want_hit=False):
        if want_hit:
            raise NotImplementedError("the restatement returns ids and Distance of primary hits, not the hit record")
        rt = self.rt
        end = W * H - 1 if end is None else end
        p = rt.make_params(W, H, mode=rt.RT_MODE_PRIMARY, traverse=rt.RT_TRAVERSE_EXACT, start=start, end=end)
        o = self.port.render(s.desc, p, nthreads=os.cpu_count() or 1, want_primary=True)
        ids = o["ids"].reshape(-1, 2)[start:end + 1]
        return dict(shape=ids[:, 0].copy(), tri=ids[:, 1].copy(), dist=o["dist"].reshape(-1)[start:end + 1].copy(), hit=None,
                    node_tests=o["counters"]["node_tests"], tri_tests=o["counters"]["tri_tests"], mismatches=0)

    def trace_rays(self, s, rays):
        return self.port.trace_rays(s.desc, rays)

    def render(self, s, W, H, mode=MODE_PATH, max_bounce=10, pass_begin=0, pass_count=1, antialias=1, seed=0,
               nthreads=1, start=0, end=None, accum=None, want_display=False):
        rt = self.rt
        self._tables(s)
        end = W * H - 1 if end is None else end
        pm = {MODE_PATH: rt.RT_MODE_PATH, MODE_PREVIEW: rt.RT_MODE_PREVIEW, MODE_WHITTED: rt.RT_MODE_WHITTED}[mode]
        p = rt.make_params(W, H, mode=pm, max_bounce=max_bounce, pass_begin=pass_begin, pass_count=pass_count,
                           antialias=antialias, seed=seed, traverse=rt.RT_TRAVERSE_EXACT, start=start, end=end)
        t0 = time.perf_counter()
        o = self.port.render(s.desc, p, nthreads=nthreads, accum=accum, want_display=want_display)
        secs = time.perf_counter() - t0
        c = o["counters"]
        # the reference's harness hands back the preview pass colour in its accum argument
        out = o["preview"] if mode == MODE_PREVIEW else o["accum"]
        return dict(accum=out, display=o["display"], seconds=secs, rays=c["rays"], shadow_rays=c["shadow_rays"])

    # -- primitive known-answer tests
    def kat_aabb(self, rays, boxes):
        return self.port.kat_aabb(rays, boxes)

    def kat_triangle(self, rays, tris):
        return self.port.kat_triangle(rays, tris)

    def kat_sphere(self, rays, spheres):
        return self.port.kat_sphere(rays, spheres)

    def kat_plane(self, rays, planes):
        return self.port.kat_plane(rays, planes)

    def kat_capsule(self, rays, caps):
        return self.port.kat_capsule(rays, caps)

    def kat_qrsqrt(self, x):
        return self.port.kat_qrsqrt(x)

    def kat_barycentric(self, pabc):
        return self.port.kat_barycentric(pabc)

    def kat_display(self, rgb):
        return self.port.kat_display(rgb)

    def kat_texture_sample(self, s, shape, slot, uv):
        return self.port.kat_texture_sample(s.mesh_texture(shape, slot), uv)
