"""ctypes mirror of include/rt_gpu.h and include/rt_host.h (struct layouts, enums, prototypes).

The C headers are authoritative; tests/test_abi.py checks that every symbol they declare is
exported by the built library and that the struct sizes here match sizeof() in C.
"""
import ctypes as C
import os

# ---- enums (include/rt_gpu.h) --------------------------------------------------------------
RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_NO_SCENE, RT_ERR_SIZE, RT_ERR_NOMEM = 0, -1, -2, -3, -4, -5
RT_SHAPE_SPHERE, RT_SHAPE_PLANE, RT_SHAPE_CAPSULE, RT_SHAPE_MESH, RT_SHAPE_TRIANGLE = range(5)
RT_MAT_DIFFUSE, RT_MAT_CHECKER, RT_MAT_REFLECTIVE, RT_MAT_EMISSIVE, RT_MAT_BLEND, RT_MAT_COMBINE, RT_MAT_NULL = range(7)
RT_LIGHT_POINT, RT_LIGHT_DIRECTIONAL = 0, 1
RT_MODE_PATH, RT_MODE_PREVIEW, RT_MODE_WHITTED, RT_MODE_PRIMARY = range(4)
RT_TRAVERSE_EXACT, RT_TRAVERSE_CULLED = 0, 1
RT_READ_ACCUM_RGBN_F32, RT_READ_DISPLAY_ARGB8, RT_READ_PRIMARY_IDS_I32X2, RT_READ_PRIMARY_DIST_F32, RT_READ_COUNTERS_U64, RT_READ_PREVIEW_RGBA_F32 = range(6)
RT_QUERY_NEAREST, RT_QUERY_ANY = 0, 1
RT_GPU_ABI_VERSION = 2
RT_GPU_FRAME_SLOTS = 4

f3 = C.c_float * 3
f2 = C.c_float * 2


class rt_shape(C.Structure):
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("has_bounds", C.c_int32), ("mesh", C.c_int32),
                ("bounds_min", f3), ("bounds_max", f3), ("a", f3), ("b", f3), ("c", f3), ("radius", C.c_float)]


class rt_material(C.Structure):
    _fields_ = [("type", C.c_int32), ("child_a", C.c_int32), ("child_b", C.c_int32), ("rgb", f3), ("scalar", C.c_float)]


class rt_bvh_node(C.Structure):
    _fields_ = [("bmin", f3), ("escape", C.c_int32), ("bmax", f3), ("tri", C.c_int32)]


class rt_tri(C.Structure):
    _fields_ = [("p0", f3), ("index", C.c_int32), ("p1", f3), ("pad0", C.c_float),
                ("p2", f3), ("pad1", C.c_float), ("n", f3), ("pad2", C.c_float)]


class rt_shade(C.Structure):
    _fields_ = [("n0", f3), ("n1", f3), ("n2", f3), ("uv0", f2), ("uv1", f2), ("uv2", f2), ("texture", C.c_int32)]


class rt_texture(C.Structure):
    _fields_ = [("rgba", C.POINTER(C.c_float)), ("width", C.c_int32), ("height", C.c_int32),
                ("texels8", C.POINTER(C.c_uint8)), ("channels", C.c_int32), ("lut", C.POINTER(C.c_float))]


class rt_mesh(C.Structure):
    _fields_ = [("nodes", C.POINTER(rt_bvh_node)), ("num_nodes", C.c_int32),
                ("tris", C.POINTER(rt_tri)), ("num_tris", C.c_int32),
                ("shade", C.POINTER(rt_shade)),
                ("textures", C.POINTER(rt_texture)), ("num_textures", C.c_int32)]


class rt_light(C.Structure):
    _fields_ = [("type", C.c_int32), ("pos_or_dir", f3), ("color", f3)]


class rt_scene_desc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32),
                ("shapes", C.POINTER(rt_shape)), ("num_shapes", C.c_int32),
                ("materials", C.POINTER(rt_material)), ("num_materials", C.c_int32),
                ("meshes", C.POINTER(rt_mesh)), ("num_meshes", C.c_int32),
                ("lights", C.POINTER(rt_light)), ("num_lights", C.c_int32),
                ("unit_vectors", C.POINTER(C.c_float)), ("num_unit_vectors", C.c_uint32),
                ("eye", f3), ("dir_z", C.c_float), ("ray_distance", C.c_float), ("bounce_offset", C.c_float)]


class rt_render_params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("start", C.c_int32), ("end", C.c_int32),
                ("mode", C.c_int32), ("max_bounce", C.c_int32), ("pass_begin", C.c_int32), ("pass_count", C.c_int32),
                ("antialias", C.c_int32), ("seed", C.c_uint32), ("traverse", C.c_int32),
                ("tile_size", C.c_int32), ("tile_count", C.c_int32), ("tile_rank", C.c_int32)]


class rt_counters(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("camera_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("node_tests", C.c_uint64), ("tri_tests", C.c_uint64),
                ("node_visits", C.c_uint64), ("tri_visits", C.c_uint64), ("mesh_hits", C.c_uint64),
                ("mesh_walks", C.c_uint64)]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_ }


class rt_ray_query(C.Structure):
    _fields_ = [("rays", C.c_void_p), ("n", C.c_int32), ("kind", C.c_int32), ("traverse", C.c_int32),
                ("shape", C.c_void_p), ("tri", C.c_void_p), ("hit", C.c_void_p)]


class rt_radiance_query(C.Structure):
    _fields_ = [("rays", C.c_void_p), ("n", C.c_int32), ("mode", C.c_int32), ("max_bounce", C.c_int32),
                ("traverse", C.c_int32), ("seed", C.c_uint32), ("sample", C.c_uint32), ("rng_stream", C.c_void_p),
                ("rng_stream_base", C.c_uint32), ("first_draw", C.c_uint32), ("rgba", C.c_void_p)]


STRUCT_SIZES = {"rt_shape": 80, "rt_material": 28, "rt_bvh_node": 32, "rt_tri": 64, "rt_shade": 64,
                "rt_light": 28, "rt_render_params": 56, "rt_counters": 72}

VP = C.c_void_p
I = C.c_int
I32 = C.c_int32
U32 = C.c_uint32
F = C.c_float
PF = C.POINTER(C.c_float)
PI32 = C.POINTER(C.c_int32)

# name -> (restype, argtypes).  Every function declared in include/rt_gpu.h and include/rt_host.h.
GPU_PROTOTYPES = {
    "rt_gpu_abi_version": (I, []),
    "rt_gpu_device_count": (I, []),
    "rt_gpu_create": (I, [I, C.POINTER(VP)]),
    "rt_gpu_destroy": (I, [VP]),
    "rt_gpu_last_error": (C.c_char_p, [VP]),
    "rt_gpu_upload_scene": (I, [VP, C.POINTER(rt_scene_desc)]),
    "rt_gpu_reset_accum": (I, [VP, I32, I32]),
    "rt_gpu_render_tile": (I, [VP, C.POINTER(rt_render_params)]),
    "rt_gpu_readback": (I, [VP, I, VP, C.c_size_t]),
    "rt_gpu_synchronize": (I, [VP]),
    "rt_gpu_last_render_ms": (I, [VP, PF]),
    "rt_gpu_last_kernel_ms": (I, [VP, PF, PI32]),
    "rt_gpu_reset_counters": (I, [VP]),
    "rt_gpu_owned_pixels": (C.c_int64, [I32, I32, I32, I32, I32]),
    "rt_gpu_pack_owned": (I, [VP, C.POINTER(rt_render_params), VP, C.c_size_t]),
    "rt_gpu_unpack_owned": (I, [VP, C.POINTER(rt_render_params), I32, VP, C.c_size_t]),
    "rt_gpu_export_frame": (I, [VP, VP, C.c_size_t]),
    "rt_gpu_open_peer_frame": (I, [VP, VP, C.c_size_t, C.POINTER(VP)]),
    "rt_gpu_close_peer_frame": (I, [VP, VP]),
    "rt_gpu_push_owned": (I, [VP, C.POINTER(rt_render_params), VP]),
    "rt_gpu_gather": (I, [C.POINTER(VP), I, I, C.POINTER(rt_render_params)]),
    "rt_gpu_resolve_display": (I, [VP]),
    "rt_gpu_stream": (VP, [VP]),
    "rt_gpu_accum_device_ptr": (VP, [VP]),
    "rt_gpu_launch_count": (C.c_uint64, [VP]),
    "rt_gpu_scene_bytes": (C.c_uint64, [VP]),
    "rt_gpu_set_tuning": (I, [VP, I32, I32, I32, I32]),
    "rt_gpu_set_pipes": (I, [VP, I32]),
    "rt_gpu_get_pipes": (I, [VP]),
    "rt_gpu_kernel_class_ms": (I, [VP, VP, VP, I32]),
    "rt_gpu_register_host_frame": (I, [VP, VP, C.c_size_t, C.POINTER(VP)]),
    "rt_gpu_unregister_host_frame": (I, [VP, VP]),
    "rt_gpu_deliver_owned": (I, [VP, C.POINTER(rt_render_params), VP, VP]),
    "rt_gpu_signal_host": (I, [VP, VP, U32]),
    "rt_gpu_set_frame_slot": (I, [VP, I32]),
    "rt_gpu_get_frame_slot": (I, [VP]),
    "rt_gpu_time_kernels": (I, [VP, I32]),
    "rt_gpu_build_bvh": (I, [VP, VP, I32, VP, I32, VP, VP, PI32, PF]),
    "rt_gpu_query_rays": (I, [VP, C.POINTER(rt_ray_query), VP]),
    "rt_gpu_radiance_rays": (I, [VP, C.POINTER(rt_radiance_query), VP]),
    "rt_gpu_trace_rays": (I, [VP, PF, I32, I32, PI32, PI32, PF]),
    "rt_gpu_kat": (I, [VP, I32, VP, VP, I32, I32, VP, VP]),
    "rt_gpu_kat_texture": (I, [VP, I32, VP, I32, VP]),
}

HOST_PROTOTYPES = {
    "rt_host_last_error": (C.c_char_p, []),
    "rt_host_scene_new": (VP, []),
    "rt_host_scene_free": (None, [VP]),
    "rt_host_mat_diffuse": (VP, [F, F, F]),
    "rt_host_mat_checker": (VP, [F, F, F, F]),
    "rt_host_mat_reflective": (VP, [F, F, F, F]),
    "rt_host_mat_emissive": (VP, [F, F, F]),
    "rt_host_mat_blend": (VP, [VP, VP, F]),
    "rt_host_mat_combine": (VP, [VP, VP]),
    "rt_host_mat_null": (VP, []),
    "rt_host_add_sphere": (I, [VP, f3, F, VP]),
    "rt_host_add_plane": (I, [VP, f3, f3, VP]),
    "rt_host_add_capsule": (I, [VP, f3, f3, F, VP]),
    "rt_host_add_triangle": (I, [VP, C.c_float * 9, VP]),
    "rt_host_add_mesh_obj": (I, [VP, C.c_char_p, VP]),
    "rt_host_add_mesh_arrays": (I, [VP, VP, I, VP, I, VP, I, VP, VP, VP, I, VP]),
    "rt_host_setup_default_scene": (I, [VP, C.c_char_p]),
    "rt_host_use_device_bvh_builder": (I, [VP]),
    "rt_host_clear_lights": (I, [VP]),
    "rt_host_add_light": (I, [VP, I, f3, f3]),
    "rt_host_set_unit_vectors": (I, [VP, U32, U32]),
    "rt_host_scene_desc": (C.POINTER(rt_scene_desc), [VP]),
    "rt_host_mesh_counts": (I, [VP, I, C.c_int32 * 7]),
    "rt_host_mesh_dump": (I, [VP, I, VP, VP, VP, VP, VP, VP, VP]),
    "rt_host_mesh_texture_info": (I, [VP, I, I, C.c_int32 * 2]),
    "rt_host_mesh_texture_pixels": (I, [VP, I, I, VP]),
    "rt_host_decode_png": (I, [C.c_char_p, C.c_int32 * 2, C.POINTER(C.c_int32), C.POINTER(C.POINTER(C.c_uint8))]),
    "rt_host_free": (None, [VP]),
    "rt_host_write_png_argb": (I, [C.c_char_p, VP, I32, I32]),
    "rt_host_program_run": (I, [VP, I, I32, I32, I32, I32, U32, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
}

LIB_NAME = "librt_b200.so"


def lib_path():
    # RT_B200_LIB selects another in-tree build of the same sources (tuning experiments only)
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), os.environ.get("RT_B200_LIB", LIB_NAME))


def bind(lib, protos):
    for name, (res, args) in protos.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    return lib
