"""raytracerwin_b200 — Python driver over the C-ABI of the B200-native RayTracerWin hot path.

Everything that computes lives in native code (raytracerwin_b200/librt_b200.so):
  * host side (C++): OBJ/MTL/PNG loading, the reference-identical BVH build, scene flattening
    (include/rt_host.h, csrc/host/);
  * device side (CUDA, sm_100a): the per-pixel ray/scene path (include/rt_gpu.h; csrc/rt_gpu.cu, rt_wave_kernels.cuh, rt_exchange.cu).
This module only marshals arguments with ctypes.  There is no CPU rendering path here: if the
library is missing, or no CUDA device is usable, construction fails loudly.
"""
import ctypes as C
import os

import numpy as np

from . import _abi
from ._abi import (rt_render_params, rt_counters, rt_scene_desc, rt_ray_query, rt_radiance_query,  # noqa: F401
                   RT_MODE_PATH, RT_MODE_PREVIEW, RT_MODE_WHITTED, RT_MODE_PRIMARY, RT_QUERY_NEAREST, RT_QUERY_ANY,
                   RT_TRAVERSE_EXACT, RT_TRAVERSE_CULLED,
                   RT_READ_ACCUM_RGBN_F32, RT_READ_DISPLAY_ARGB8, RT_READ_PRIMARY_IDS_I32X2,
                   RT_READ_PRIMARY_DIST_F32, RT_READ_COUNTERS_U64, RT_READ_PREVIEW_RGBA_F32)

_lib = None


class RtError(RuntimeError):
    pass


def load_library():
    """Loads librt_b200.so (built by __graft_entry__.build()).  Raises if it is absent."""
    global _lib
    if _lib is None:
        path = _abi.lib_path()
        if not os.path.exists(path):
            raise RtError(f"{path} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback for the render path)")
        lib = C.CDLL(path)
        _abi.bind(lib, _abi.GPU_PROTOTYPES)
        _abi.bind(lib, _abi.HOST_PROTOTYPES)
        _lib = lib
    return _lib


# ---- material / shape specs --------------------------------------------------------------------
# A scene is described by plain tuples so that the same description can be fed to this package
# and, in tests, to the reference oracle:
#   material: ("diffuse", rgb) | ("checker", rgb, size) | ("reflective", rgb, fuzz) | ("emissive", rgb)
#             | ("blend", A, B, factor) | ("combine", A, B) | ("null",) | None
#   shape:    ("sphere", center, radius, mat) | ("plane", normal, point, mat)
#             | ("capsule", start, end, radius, mat) | ("triangle", p0, p1, p2, mat) | ("mesh", obj_path, mat)

def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def _make_material(lib, spec):
    if spec is None:
        return None
    kind = spec[0]
    if kind == "diffuse":
        return lib.rt_host_mat_diffuse(*map(float, spec[1]))
    if kind == "checker":
        return lib.rt_host_mat_checker(*map(float, spec[1]), float(spec[2]))
    if kind == "reflective":
        return lib.rt_host_mat_reflective(*map(float, spec[1]), float(spec[2]))
    if kind == "emissive":
        return lib.rt_host_mat_emissive(*map(float, spec[1]))
    if kind == "blend":
        return lib.rt_host_mat_blend(_make_material(lib, spec[1]), _make_material(lib, spec[2]), float(spec[3]))
    if kind == "combine":
        return lib.rt_host_mat_combine(_make_material(lib, spec[1]), _make_material(lib, spec[2]))
    if kind == "null":
        return lib.rt_host_mat_null()
    raise ValueError(f"unknown material {kind!r}")


class Scene:
    """RayTracerScene: AddShape(shape, material) on the host, flattened for the device."""

    def __init__(self, shapes=()):
        self._lib = load_library()
        self._h = self._lib.rt_host_scene_new()
        for s in shapes:
            self.add(s)

    def close(self):
        if self._h:
            self._lib.rt_host_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise RtError(self._lib.rt_host_last_error().decode() or f"rt_host error {rc}")
        return rc

    def add(self, spec):
        lib, kind = self._lib, spec[0]
        mat = _make_material(lib, spec[-1])
        if kind == "sphere":
            return self._check(lib.rt_host_add_sphere(self._h, _f3(spec[1]), float(spec[2]), mat))
        if kind == "plane":
            return self._check(lib.rt_host_add_plane(self._h, _f3(spec[1]), _f3(spec[2]), mat))
        if kind == "capsule":
            return self._check(lib.rt_host_add_capsule(self._h, _f3(spec[1]), _f3(spec[2]), float(spec[3]), mat))
        if kind == "triangle":
            p = (C.c_float * 9)(*[float(x) for v in spec[1:4] for x in v])
            return self._check(lib.rt_host_add_triangle(self._h, p, mat))
        if kind == "mesh":
            return self._check(lib.rt_host_add_mesh_obj(self._h, os.fsencode(spec[1]), mat))
        if kind == "mesh_arrays":
            return self.add_mesh_arrays(*spec[1:-1], material=spec[-1], _mat_handle=mat)
        raise ValueError(f"unknown shape {kind!r}")

    def add_mesh_arrays(self, points, point_idx, normals=None, normal_idx=None, texcoords=None,
                        texcoord_idx=None, material=None, _mat_handle=None):
        lib = self._lib
        mat = _mat_handle if _mat_handle is not None else _make_material(lib, material)
        pts = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
        pidx = np.ascontiguousarray(point_idx, np.int32).reshape(-1, 3)
        nrm = None if normals is None else np.ascontiguousarray(normals, np.float32).reshape(-1, 3)
        nidx = None if normal_idx is None else np.ascontiguousarray(normal_idx, np.int32).reshape(-1, 3)
        tex = None if texcoords is None else np.ascontiguousarray(texcoords, np.float32).reshape(-1, 2)
        tidx = None if texcoord_idx is None else np.ascontiguousarray(texcoord_idx, np.int32).reshape(-1, 3)
        ptr = lambda a: None if a is None else a.ctypes.data
        return self._check(lib.rt_host_add_mesh_arrays(
            self._h, ptr(pts), len(pts), ptr(nrm), 0 if nrm is None else len(nrm),
            ptr(tex), 0 if tex is None else len(tex), ptr(pidx), ptr(nidx), ptr(tidx), len(pidx), mat))

    def setup_default_scene(self, data_dir):
        """RayTracerProgram::SetupScene (RayTracerProgram.cpp:467-552)."""
        self._check(self._lib.rt_host_setup_default_scene(self._h, os.fsencode(data_dir)))

    def set_unit_vectors(self, seed=0, count=0):
        """PseudoRandomUnitVectors table for Diffuse materials; count=0 -> the reference's 0xFFFFFF."""
        self._check(self._lib.rt_host_set_unit_vectors(self._h, seed, count))

    def set_lights(self, lights):
        self._lib.rt_host_clear_lights(self._h)
        for kind, v, color in lights:
            self._lib.rt_host_add_light(self._h, int(kind), _f3(v), _f3(color))

    @property
    def desc(self):
        """POINTER(rt_scene_desc) valid until the scene changes."""
        return self._lib.rt_host_scene_desc(self._h)

    # -- introspection used by the loader/BVH parity tests
    def mesh_counts(self, shape):
        out = (C.c_int32 * 7)()
        self._check(self._lib.rt_host_mesh_counts(self._h, shape, out))
        return list(out)

    def mesh_dump(self, shape):
        npts, ntex, nnrm, ntri, _, _, _ = self.mesh_counts(shape)
        d = dict(points=np.zeros((npts, 3), np.float32), texcoords=np.zeros((ntex, 3), np.float32),
                 normals=np.zeros((nnrm, 3), np.float32), pidx=np.zeros(3 * ntri, np.int32),
                 tidx=np.zeros(3 * ntri, np.int32), nidx=np.zeros(3 * ntri, np.int32), matid=np.zeros(ntri, np.int32))
        self._check(self._lib.rt_host_mesh_dump(self._h, shape, *[d[k].ctypes.data for k in
                                                               ("points", "texcoords", "normals", "pidx", "tidx", "nidx", "matid")]))
        return d

    def mesh_texture(self, shape, slot):
        wh = (C.c_int32 * 2)()
        self._check(self._lib.rt_host_mesh_texture_info(self._h, shape, slot, wh))
        if wh[0] == 0:
            return None
        px = np.zeros((wh[1], wh[0], 4), np.float32)
        self._check(self._lib.rt_host_mesh_texture_pixels(self._h, shape, slot, px.ctypes.data))
        return px

    def flat_mesh(self, mesh_index=0):
        """numpy copies of the flattened mesh arrays in the scene description."""
        m = self.desc.contents.meshes[mesh_index]
        nodes = np.ctypeslib.as_array(C.cast(m.nodes, C.POINTER(C.c_uint8)), (m.num_nodes * 32,)).copy()
        tris = np.ctypeslib.as_array(C.cast(m.tris, C.POINTER(C.c_uint8)), (m.num_tris * 64,)).copy()
        shade = np.ctypeslib.as_array(C.cast(m.shade, C.POINTER(C.c_uint8)), (m.num_tris * 64,)).copy()
        node_dt = np.dtype([("bmin", "<f4", 3), ("escape", "<i4"), ("bmax", "<f4", 3), ("tri", "<i4")])
        tri_dt = np.dtype([("p0", "<f4", 3), ("index", "<i4"), ("p1", "<f4", 3), ("pad0", "<f4"),
                           ("p2", "<f4", 3), ("pad1", "<f4"), ("n", "<f4", 3), ("pad2", "<f4")])
        shade_dt = np.dtype([("n0", "<f4", 3), ("n1", "<f4", 3), ("n2", "<f4", 3),
                             ("uv0", "<f4", 2), ("uv1", "<f4", 2), ("uv2", "<f4", 2), ("texture", "<i4")])
        return nodes.view(node_dt), tris.view(tri_dt), shade.view(shade_dt)


def use_device_bvh_builder(ctx):
    """Meshes loaded from now on get their tree built on `ctx`'s GPU (None: back to the host builder)."""
    load_library().rt_host_use_device_bvh_builder(ctx.handle if ctx is not None else None)


def make_params(width, height, mode=RT_MODE_PATH, max_bounce=10, pass_begin=0, pass_count=1,
                antialias=1, seed=0, traverse=RT_TRAVERSE_CULLED, start=0, end=None,
                tile_size=0, tile_count=0, tile_rank=0):
    p = rt_render_params()
    p.width, p.height = width, height
    p.start = start
    p.end = width * height - 1 if end is None else end
    p.mode, p.max_bounce = mode, max_bounce
    p.pass_begin, p.pass_count = pass_begin, pass_count
    p.antialias, p.seed, p.traverse = antialias, seed, traverse
    p.tile_size, p.tile_count, p.tile_rank = tile_size, tile_count, tile_rank
    return p


class GpuContext:
    """One rt_gpu_ctx: a scene resident on one B200 plus its device framebuffers."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.rt_gpu_create(device, C.byref(h))
        if rc != 0:
            raise RtError(f"rt_gpu_create({device}) failed: {self._lib.rt_gpu_last_error(None).decode()}")
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rt_gpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RtError(f"rt_gpu error {rc}: {self._lib.rt_gpu_last_error(self._h).decode()}")

    @property
    def handle(self):
        return self._h

    def upload_scene(self, scene):
        desc = scene.desc if isinstance(scene, Scene) else scene
        self._check(self._lib.rt_gpu_upload_scene(self._h, desc))

    def reset_accum(self, width, height):
        self._check(self._lib.rt_gpu_reset_accum(self._h, width, height))

    def reset_counters(self):
        self._check(self._lib.rt_gpu_reset_counters(self._h))

    def render_tile(self, params):
        self._check(self._lib.rt_gpu_render_tile(self._h, C.byref(params)))

    def synchronize(self):
        self._check(self._lib.rt_gpu_synchronize(self._h))

    def last_render_ms(self):
        ms = C.c_float()
        self._check(self._lib.rt_gpu_last_render_ms(self._h, C.byref(ms)))
        return ms.value

    def last_kernel_ms(self):
        """(ms inside the path kernel during the last render_tile, number of its launches)"""
        ms, n = C.c_float(), C.c_int32()
        self._check(self._lib.rt_gpu_last_kernel_ms(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def set_tuning(self, window_items=32, min_lanes=28, leaf_wait=18, pool_kpaths=0):
        self._check(self._lib.rt_gpu_set_tuning(self._h, window_items, min_lanes, leaf_wait, pool_kpaths))

    def time_kernels(self, on=True):
        """True / 1: an event pair around every walk bracket; 2: one event per launch, by kernel class."""
        self._check(self._lib.rt_gpu_time_kernels(self._h, int(on)))

    KERNEL_CLASSES = ("generate", "packet_walk", "walk", "long_walk", "shade", "fold", "other")

    def kernel_class_ms(self):
        """{class: (ms, launches)} of the last render_tile made under time_kernels(2)."""
        n = len(self.KERNEL_CLASSES)
        ms, cnt = (C.c_float * n)(), (C.c_int32 * n)()
        self._check(self._lib.rt_gpu_kernel_class_ms(self._h, ms, cnt, n))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.KERNEL_CLASSES)}

    def set_pipes(self, pipes):
        """Concurrent pass-chunk streams of a render call (0 restores the default)."""
        self._check(self._lib.rt_gpu_set_pipes(self._h, pipes))

    def set_frame_slot(self, slot):
        """Address the other set of frame buffers (own stream): frames on different slots overlap on the device."""
        self._check(self._lib.rt_gpu_set_frame_slot(self._h, slot))

    def get_pipes(self):
        return int(self._lib.rt_gpu_get_pipes(self._h))

    @property
    def launch_count(self):
        return int(self._lib.rt_gpu_launch_count(self._h))

    def readback(self, what, width, height, out=None):
        if what in (RT_READ_ACCUM_RGBN_F32, RT_READ_PREVIEW_RGBA_F32):
            out = np.empty((height, width, 4), np.float32) if out is None else out
        elif what == RT_READ_DISPLAY_ARGB8:
            out = np.empty((height, width), np.uint32) if out is None else out
        elif what == RT_READ_PRIMARY_IDS_I32X2:
            out = np.empty((height, width, 2), np.int32) if out is None else out
        elif what == RT_READ_PRIMARY_DIST_F32:
            out = np.empty((height, width), np.float32) if out is None else out
        else:
            raise ValueError(what)
        self._check(self._lib.rt_gpu_readback(self._h, what, out.ctypes.data, out.nbytes))
        return out

    def readback_into(self, what, ptr, nbytes):
        self._check(self._lib.rt_gpu_readback(self._h, what, ptr, nbytes))

    def counters(self):
        c = rt_counters()
        self._check(self._lib.rt_gpu_readback(self._h, RT_READ_COUNTERS_U64, C.byref(c), C.sizeof(c)))
        return c.as_dict()

    def trace_rays(self, rays, traverse=RT_TRAVERSE_EXACT):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = len(rays)
        shape = np.empty(n, np.int32)
        tri = np.empty(n, np.int32)
        hit = np.empty((n, 11), np.float32)
        self._check(self._lib.rt_gpu_trace_rays(
            self._h, rays.ctypes.data_as(_abi.PF), n, traverse,
            shape.ctypes.data_as(_abi.PI32), tri.ctypes.data_as(_abi.PI32), hit.ctypes.data_as(_abi.PF)))
        return shape, tri, hit

    def _device_tensor(self, name, t, dtype, shape):
        """Checks that `t` is a contiguous torch tensor of `dtype` and `shape` (None = any length) on this GPU."""
        import torch
        dev = torch.device("cuda", self.device)
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"{name} must be a torch tensor on {dev}, not {type(t).__name__}")
        if t.device != dev:
            raise ValueError(f"{name} on {t.device}, but the context is on {dev}")
        if t.dtype != dtype:
            raise ValueError(f"{name} must be {dtype}, not {t.dtype}")
        if t.dim() != len(shape) or any(s is not None and t.shape[k] != s for k, s in enumerate(shape)):
            want = tuple("N" if s is None else s for s in shape)
            raise ValueError(f"{name} must have shape {want}, not {tuple(t.shape)}")
        if not t.is_contiguous():
            raise ValueError(f"{name} must be contiguous")

    @staticmethod
    def _torch_stream(dev):
        import torch
        # torch names the legacy default stream 0, which the C calls would take for the context's own stream:
        # pass it as cudaStreamLegacy (1) instead
        return torch.cuda.current_stream(dev).cuda_stream or 1

    def query_rays(self, rays, any_hit=False, traverse=RT_TRAVERSE_CULLED, want_tri=None, want_hit=None):
        """Nearest-hit or occlusion queries of a batch of rays held in device memory (rt_gpu_query_rays).

        `rays`: contiguous float32 torch tensor (N, 7) {origin, direction, Distance} on cuda:<self.device>.
        The queries are enqueued on torch.cuda.current_stream(self.device) and the call returns at once; the
        results are usable on that stream without a host synchronisation.  Outputs are torch tensors on the same
        device: nearest hit -> dict(shape=int32[N] (-1 = none), tri=int32[N] or None, hit=float32[N, 11] or None)
        with rt_gpu_trace_rays' fields; any_hit -> int32[N], 1 where the ray is occluded.  want_tri / want_hit
        default to True for nearest-hit queries and to False for occlusion queries (which have neither).
        The context's counters are read on its own stream: synchronise before reading them."""
        import torch
        self._device_tensor("rays", rays, torch.float32, (None, 7))
        dev = torch.device("cuda", self.device)
        n = rays.shape[0]
        want_tri = not any_hit if want_tri is None else want_tri
        want_hit = not any_hit if want_hit is None else want_hit
        shape = torch.empty(n, dtype=torch.int32, device=dev)
        tri = torch.empty(n, dtype=torch.int32, device=dev) if want_tri else None
        hit = torch.empty((n, 11), dtype=torch.float32, device=dev) if want_hit else None
        q = rt_ray_query(rays.data_ptr(), n, RT_QUERY_ANY if any_hit else RT_QUERY_NEAREST, traverse, shape.data_ptr(),
                         None if tri is None else tri.data_ptr(), None if hit is None else hit.data_ptr())
        self._check(self._lib.rt_gpu_query_rays(self._h, C.byref(q), self._torch_stream(dev)))
        if any_hit:
            return shape
        return dict(shape=shape, tri=tri, hit=hit)

    def radiance_rays(self, rays, mode=RT_MODE_PATH, max_bounce=10, seed=0, sample=0, rng_stream=None,
                      rng_stream_base=0, first_draw=0, traverse=RT_TRAVERSE_CULLED, out=None):
        """Radiance of a batch of rays held in device memory (rt_gpu_radiance_rays): RayTrace's path (RT_MODE_PATH), its
        preview colour (RT_MODE_PREVIEW) or the Whitted composition (RT_MODE_WHITTED) of each ray, as render_tile
        computes it for a camera ray.

        `rays`: contiguous float32 torch tensor (N, 7) {origin, direction, Distance} on cuda:<self.device>.  Ray i draws
        its random numbers from rt_rng_key(seed, stream_i, sample) starting at draw `first_draw`, with stream_i =
        rng_stream[i] (an int32 (N,) tensor on the same device whose bits are the stream ids) or rng_stream_base + i.
        `out`: optional contiguous float32 (N, 4) tensor on the same device to write into.  Enqueued on
        torch.cuda.current_stream(self.device); returns the float32 (N, 4) tensor {r, g, b, 0}, usable on that stream
        without a host synchronisation.  The context's counters are read on its own stream: synchronise before
        reading them."""
        import torch
        self._device_tensor("rays", rays, torch.float32, (None, 7))
        dev = torch.device("cuda", self.device)
        n = rays.shape[0]
        if rng_stream is not None:
            self._device_tensor("rng_stream", rng_stream, torch.int32, (n,))
        if out is None:
            out = torch.empty((n, 4), dtype=torch.float32, device=dev)
        else:
            self._device_tensor("out", out, torch.float32, (n, 4))
        q = rt_radiance_query(rays.data_ptr(), n, mode, max_bounce, traverse, seed & 0xFFFFFFFF, sample & 0xFFFFFFFF,
                              None if rng_stream is None else rng_stream.data_ptr(), rng_stream_base & 0xFFFFFFFF,
                              first_draw & 0xFFFFFFFF, out.data_ptr())
        self._check(self._lib.rt_gpu_radiance_rays(self._h, C.byref(q), self._torch_stream(dev)))
        return out

    def build_bvh(self, points, point_idx):
        """KdTree::Build on the device: (nodes, tris, depth, device ms) with the dtypes of Scene.flat_mesh."""
        pts = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
        idx = np.ascontiguousarray(point_idx, np.int32).reshape(-1, 3)
        n = len(idx)
        node_dt = np.dtype([("bmin", "<f4", 3), ("escape", "<i4"), ("bmax", "<f4", 3), ("tri", "<i4")])
        tri_dt = np.dtype([("p0", "<f4", 3), ("index", "<i4"), ("p1", "<f4", 3), ("pad0", "<f4"),
                           ("p2", "<f4", 3), ("pad1", "<f4"), ("n", "<f4", 3), ("pad2", "<f4")])
        nodes = np.zeros(2 * n - 1, node_dt)
        tris = np.zeros(n, tri_dt)
        depth, ms = C.c_int32(), C.c_float()
        self._check(self._lib.rt_gpu_build_bvh(self._h, pts.ctypes.data, len(pts), idx.ctypes.data, n,
                                               nodes.ctypes.data, tris.ctypes.data, C.byref(depth), C.byref(ms)))
        return nodes, tris, depth.value, ms.value

    def pack_owned(self, params, dev_ptr, nbytes):
        self._check(self._lib.rt_gpu_pack_owned(self._h, C.byref(params), dev_ptr, nbytes))

    def unpack_owned(self, params, src_rank, dev_ptr, nbytes):
        self._check(self._lib.rt_gpu_unpack_owned(self._h, C.byref(params), src_rank, dev_ptr, nbytes))

    def register_host_frame(self, host_ptr, nbytes):
        """Pin + map caller host memory (e.g. a shared-memory frame) into this GPU; returns the device address."""
        out = C.c_void_p()
        self._check(self._lib.rt_gpu_register_host_frame(self._h, host_ptr, nbytes, C.byref(out)))
        return out.value

    def unregister_host_frame(self, host_ptr):
        self._check(self._lib.rt_gpu_unregister_host_frame(self._h, host_ptr))

    def deliver_owned(self, params, host_accum_dev, host_display_dev):
        """This rank's owned tiles of accuBuffer / bitcolor written straight into registered host frames."""
        self._check(self._lib.rt_gpu_deliver_owned(self._h, C.byref(params), host_accum_dev, host_display_dev))

    def signal_host(self, host_word_dev, value):
        """Stream-ordered write of a 32-bit word of a registered host frame (e.g. 'this rank delivered frame k')."""
        self._check(self._lib.rt_gpu_signal_host(self._h, host_word_dev, value))

    def export_frame(self):
        """64-byte CUDA IPC handle of the accumulation buffer (bytes); call after reset_accum."""
        buf = C.create_string_buffer(64)
        self._check(self._lib.rt_gpu_export_frame(self._h, buf, 64))
        return buf.raw

    def open_peer_frame(self, handle):
        """Maps another process's exported accumulation buffer; returns its device address on this GPU."""
        buf = C.create_string_buffer(bytes(handle), 64)
        out = C.c_void_p()
        self._check(self._lib.rt_gpu_open_peer_frame(self._h, buf, 64, C.byref(out)))
        return out.value

    def close_peer_frame(self, dev_ptr):
        self._check(self._lib.rt_gpu_close_peer_frame(self._h, dev_ptr))

    def push_owned(self, params, peer_frame):
        self._check(self._lib.rt_gpu_push_owned(self._h, C.byref(params), peer_frame))

    def resolve_display(self):
        self._check(self._lib.rt_gpu_resolve_display(self._h))

    @property
    def stream(self):
        return self._lib.rt_gpu_stream(self._h)


def owned_pixels(width, height, tile_size, tile_count, tile_rank):
    return int(load_library().rt_gpu_owned_pixels(width, height, tile_size, tile_count, tile_rank))
