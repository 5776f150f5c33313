/* rt_host.h — C handle API over the host-side (CPU, C++) scene layer.
 *
 * The scene layer itself is C++ (raytracerwin_b200/csrc/host/rt_host.hpp) and mirrors the
 * reference's public surface for this path: RayTracerScene::AddShape (RayTracerScene.h:49),
 * RMeshShape::Create (MeshShape.h:23), RSphere/RPlane/RCapsule::Create (Shapes.h:58,74,96) and the
 * seven SurfaceMaterial_* classes (SurfaceMaterials.h:48-141).  These C entry points exist so that
 * Python (tests/, bench.py) can build the same scenes through ctypes; a C++ embedder uses the
 * classes directly.  Everything here runs on the CPU: OBJ/MTL/PNG loading, the BVH build with the
 * reference's partition rule (KdTree.cpp:37-126) and the flattening into rt_scene_desc.
 */
#ifndef RT_HOST_H
#define RT_HOST_H

#include "rt_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rt_host_scene rt_host_scene;       /* RayTracerScene */
typedef struct rt_host_material rt_host_material; /* ISurfaceMaterial (ownership moves on use) */

const char* rt_host_last_error(void);

rt_host_scene* rt_host_scene_new(void);
void rt_host_scene_free(rt_host_scene* s);

/* SurfaceMaterial_* constructors, SurfaceMaterials.cpp:15,40,92,127,145,163 / .h:134 */
rt_host_material* rt_host_mat_diffuse(float r, float g, float b);
rt_host_material* rt_host_mat_checker(float r, float g, float b, float pattern_size);
rt_host_material* rt_host_mat_reflective(float r, float g, float b, float fuzziness);
rt_host_material* rt_host_mat_emissive(float r, float g, float b);
rt_host_material* rt_host_mat_blend(rt_host_material* a, rt_host_material* b, float factor);
rt_host_material* rt_host_mat_combine(rt_host_material* a, rt_host_material* b);
rt_host_material* rt_host_mat_null(void);

/* RayTracerScene::AddShape(Shape::Create(...), material); return the shape index or <0.
 * `mat` may be NULL (shape without material) and is consumed. */
int rt_host_add_sphere(rt_host_scene* s, const float center[3], float radius, rt_host_material* mat);
int rt_host_add_plane(rt_host_scene* s, const float normal[3], const float point[3], rt_host_material* mat);
int rt_host_add_capsule(rt_host_scene* s, const float start[3], const float end[3], float radius, rt_host_material* mat);
int rt_host_add_triangle(rt_host_scene* s, const float p[9], rt_host_material* mat);
int rt_host_add_mesh_obj(rt_host_scene* s, const char* obj_path, rt_host_material* mat);
/* Mesh from memory: positions/normals xyz triples, texcoords uv pairs, per-corner indices
 * (3 per triangle), no textures.  normals/texcoords (and their indices) may be NULL: the flat
 * face normal / zero uv are used. */
int rt_host_add_mesh_arrays(rt_host_scene* s, const float* points, int num_points,
                            const float* normals, int num_normals,
                            const float* texcoords, int num_texcoords,
                            const int32_t* point_idx, const int32_t* normal_idx,
                            const int32_t* texcoord_idx, int num_tris, rt_host_material* mat);

/* The reference's hard-coded scene, RayTracerProgram::SetupScene (RayTracerProgram.cpp:467-552);
 * `data_dir` is the directory that holds unitychan.obj. */
int rt_host_setup_default_scene(rt_host_scene* s, const char* data_dir);

/* Meshes added after this call get their tree from rt_gpu_build_bvh on `ctx` (KdTree::Build on the device,
 * identical arrays); NULL switches back to the host builder.  Process-wide, not thread-safe. */
int rt_host_use_device_bvh_builder(rt_gpu_ctx* ctx);

/* Lights default to the reference's GSceneLights (RayTracerScene.cpp:14-18) */
int rt_host_clear_lights(rt_host_scene* s);
int rt_host_add_light(rt_host_scene* s, int type, const float pos_or_dir[3], const float color[3]);

/* PseudoRandomUnitVectors (Math.cpp:17-31): `count` entries generated from the counter RNG
 * stream (seed, RT_RNG_TABLE_PIXEL, 0).  count = 0 selects the reference's 0xFFFFFF. */
int rt_host_set_unit_vectors(rt_host_scene* s, uint32_t seed, uint32_t count);

/* Flattened view of the scene; owned by the scene, valid until it is modified or freed. */
const rt_scene_desc* rt_host_scene_desc(rt_host_scene* s);

/* Introspection of a loaded mesh (pins the loader/BVH builder against the reference). */
/* out = {points, texcoords, normals, triangles, material slots, bvh nodes, bvh depth} */
int rt_host_mesh_counts(rt_host_scene* s, int shape, int32_t out[7]);
int rt_host_mesh_dump(rt_host_scene* s, int shape, float* points, float* texcoords, float* normals,
                      int32_t* pidx, int32_t* tidx, int32_t* nidx, int32_t* matid);
/* material slot -> {width,height} (0,0 when the slot has no texture); pixels = RGBA float */
int rt_host_mesh_texture_info(rt_host_scene* s, int shape, int slot, int32_t wh[2]);
int rt_host_mesh_texture_pixels(rt_host_scene* s, int shape, int slot, float* out);

/* Stand-alone helpers */
/* The 512-entry table of rt_texture.lut that the PNG loader builds (lut[c] = powf(c / 255, 2.2f) by this host's powf,
 * lut[256 + c] = c / 255): 8-bit texels fed through it to rt_gpu_update_texture equal the loader's texels bit for bit. */
int rt_host_texel_lut(float* out512);
int rt_host_decode_png(const char* path, int32_t wh[2], int32_t* channels, uint8_t** out_pixels);
void rt_host_free(void* p);
int rt_host_write_png_argb(const char* path, const uint32_t* argb, int32_t width, int32_t height);

/* Headless RayTracerProgram::Run (RayTracerProgram.cpp:270-422,437-456): preview pass, then
 * `passes` accumulation passes on GPU `device`, optional PNG of the display buffer. */
int rt_host_program_run(rt_host_scene* s, int device, int32_t width, int32_t height,
                        int32_t passes, int32_t max_bounce, uint32_t seed, const char* png_path,
                        double* out_seconds, uint64_t* out_rays);

#ifdef __cplusplus
}
#endif
#endif /* RT_HOST_H */
