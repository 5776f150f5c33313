/* rt_gpu.h — C-ABI boundary of the B200-native per-pixel ray/scene hot path.
 *
 * The reference (aosyang/RayTracerWin) has no plugin/FFI interface; its seam for this path is
 * the per-task call  ThreadWorker_Render(Task.Start, Task.End, MaxBounceTimes, Task.Option)
 * (Src/RayTracerProgram.cpp:131, called from ThreadTaskWorker at :235, tasks pushed at
 * :294-302 and :320-327), which reads the scene through a singleton (:134) and writes the
 * file-scope globals bitcolor[] (:49) and accuBuffer[] (:77).  This header makes every one of
 * those implicit inputs/outputs explicit:
 *
 *   rt_gpu_upload_scene  replaces the implicit read of RayTracerProgram::GetScene() (:134),
 *                        the camera constants (:133,:141-142,:164), GSceneLights
 *                        (RayTracerScene.cpp:14-18) and PseudoRandomUnitVectors (Math.cpp:17-19)
 *   rt_gpu_render_tile   replaces ThreadWorker_Render(begin, end, MaxBounceCount, Option)
 *                        (RayTracerProgram.cpp:131-188), i.e. one RenderThreadTask (:79-95)
 *   rt_gpu_render_view   render_tile from a camera of the call's own: eye, orientation and image plane per call
 *   rt_gpu_readback      replaces reading bitcolor[] / accuBuffer[] (:49,:77)
 *   rt_gpu_query_rays    FindIntersectionWithScene (RayTracerScene.cpp:99-125) and the shadow query of
 *                        CalculateLightColor (:152-164) on batches of the caller's rays in device memory
 *   rt_gpu_radiance_rays RayTracerScene::RayTrace (RayTracerScene.cpp:31-97), its preview branch, or the Whitted
 *                        composition, on batches of the caller's rays in device memory (own cameras, probes, bakes)
 *   rt_gpu_update_mesh   new mesh geometry from device memory (tree rebuilt on the device) and moved analytic
 *   rt_gpu_update_shapes shapes, without a new upload and without draining frames in flight
 *   rt_gpu_refit_mesh    new points under a mesh's published tree (boxes recomputed, topology kept), with no host wait
 *   rt_gpu_replace_mesh  a new mesh of any triangle count, with texture coordinates and texture slots, from device memory
 *                        (levels of detail, procedural and streamed geometry) without a new upload
 *   rt_gpu_update_materials  material nodes edited in place or appended, rt_gpu_update_lights a new light list and
 *   rt_gpu_update_texture    a rectangle of texels from device memory: the scene's appearance without a new upload
 *   rt_gpu_track_moments     per-pixel moments of the pass colours (the error estimate of each pixel of a frame slot),
 *   rt_gpu_select_pixels     the pixels whose estimate is above a tolerance, as a device mask, and
 *   rt_gpu_render_masked     render_tile restricted to a device pixel mask: adaptive sampling
 *   rt_gpu_denoise           an edge-avoiding a-trous filter of a frame slot's mean colour, guided by the first-hit ids,
 *                            distances and normals of an RT_MODE_GUIDES render, into the caller's device memory
 *
 * Plain C: POD structs, pointers and sizes only.  No C++/STL/torch types cross the boundary.
 * Every entry returns 0 on success or a negative rt_status; rt_gpu_last_error() gives text.
 * A context is bound to one GPU and is not thread-safe (one host thread per context).
 * There is NO CPU fallback: if no CUDA device is usable rt_gpu_create fails with RT_ERR_CUDA.
 */
#ifndef RT_GPU_H
#define RT_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_GPU_ABI_VERSION 2

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1,   /* bad argument / malformed scene */
    RT_ERR_CUDA = -2,      /* CUDA runtime error (text in rt_gpu_last_error) */
    RT_ERR_NO_SCENE = -3,  /* render/readback before upload */
    RT_ERR_SIZE = -4,      /* readback buffer too small */
    RT_ERR_NOMEM = -5
} rt_status;

/* ---- scene description (all host pointers; upload copies everything) ------------------ */

/* RShape subclasses, Src/Shapes.h:46,64,82,104 and Src/MeshShape.h:16 */
enum { RT_SHAPE_SPHERE = 0, RT_SHAPE_PLANE = 1, RT_SHAPE_CAPSULE = 2, RT_SHAPE_MESH = 3,
       RT_SHAPE_TRIANGLE = 4 };

/* ISurfaceMaterial subclasses, Src/SurfaceMaterials.h:48-141 */
enum { RT_MAT_DIFFUSE = 0, RT_MAT_CHECKER = 1, RT_MAT_REFLECTIVE = 2, RT_MAT_EMISSIVE = 3,
       RT_MAT_BLEND = 4, RT_MAT_COMBINE = 5, RT_MAT_NULL = 6 };

/* ELightType, Src/Light.h:10-14 */
enum { RT_LIGHT_POINT = 0, RT_LIGHT_DIRECTIONAL = 1 };

typedef struct rt_shape {
    int32_t type;           /* RT_SHAPE_* */
    int32_t material;       /* root node in materials[], -1 = no material (RShape::SurfaceMaterial null) */
    int32_t has_bounds;     /* RShape::HasCullingBounds(): 0 for planes (Shapes.cpp:28) */
    int32_t mesh;           /* index into meshes[] for RT_SHAPE_MESH, else -1 */
    float bounds_min[3];    /* RShape::Aabb */
    float bounds_max[3];
    float a[3];             /* sphere Center | plane Normal | capsule Start | triangle p0 */
    float b[3];             /* plane Point | capsule End | triangle p1 */
    float c[3];             /* triangle p2 */
    float radius;           /* sphere / capsule Radius */
} rt_shape;

/* One node of a material graph (Blend/Combine reference children by index; nodes may be shared).  rt_gpu_upload_scene
 * refuses (RT_ERR_INVALID) a graph with a cycle and one in which some path from ANY node down to a leaf passes more
 * than 8 Combine nodes (the device's frame stack of Combines; Blend nodes do not count), whether or not a shape uses
 * that node, since rt_gpu_update_shapes may point a shape at it later. */
typedef struct rt_material {
    int32_t type;           /* RT_MAT_* */
    int32_t child_a;        /* Blend: BlendMaterialA, Combine: MaterialA; else -1 */
    int32_t child_b;
    float rgb[3];           /* Albedo / emissive Color */
    float scalar;           /* Checker: ReciprocalPatternSize; Reflective: Fuzziness; Blend: BlendFactor */
} rt_material;

/* Pre-order ("threaded") flattening of the reference's KdNode tree (Src/KdTree.h:64-77):
 * node i's left child is i+1; `escape` is the next node in pre-order that is not in i's
 * subtree (== num_nodes at the end).  Visiting "hit -> i+1, miss or leaf -> escape" reproduces
 * KdNode::TestRayIntersection's fixed Left-then-Right order (KdTree.cpp:128-195) with no stack. */
typedef struct rt_bvh_node {
    float bmin[3];          /* KdNode::Bounds.pMin */
    int32_t escape;
    float bmax[3];          /* KdNode::Bounds.pMax */
    int32_t tri;            /* leaf: index into rt_mesh.tris (leaf order); inner: -1 */
} rt_bvh_node;              /* 32 B = two 16-byte loads */

/* One leaf triangle, in leaf (pre-order) order.  `n` is the face normal exactly as
 * RRay::TestIntersectionWithTriangle computes it per test (RRay.cpp:138-145):
 * cross(p1-p0,p2-p0).GetNormalizedVec3(), host-precomputed without FP contraction. */
typedef struct rt_tri {
    float p0[3]; int32_t index;   /* TriangleData::Index = triangle id in the original mesh */
    float p1[3]; float pad0;
    float p2[3]; float pad1;
    float n[3];  float pad2;
} rt_tri;                   /* 64 B = four 16-byte loads */

/* Per-triangle shading attributes in ORIGINAL triangle order (MeshShape.cpp:286-326). */
typedef struct rt_shade {
    float n0[3], n1[3], n2[3];    /* Normals[NormalIndices[3t+k]] */
    float uv0[2], uv1[2], uv2[2]; /* Texcoords[TexcoordIndices[3t+k]].xy */
    int32_t texture;              /* index into rt_mesh.textures, -1 = untextured
                                     (MaterialId == -1, out of range, or Textures[id] null) */
} rt_shade;                 /* 64 B */

typedef struct rt_texture {
    const float* rgba;      /* width*height RVec4 texels, linear-light rgb (Texture.cpp:130,147) — or NULL when the
                               texture comes as 8-bit texels below (NULL in both: an empty slot) */
    int32_t width, height;
    /* The decoded PNG as it is (`channels` = 3 or 4 bytes per texel) plus the 512-entry table that turns a code into
     * the reference's texel: lut[c] = powf(c / 255, 2.2f) for r, g, b (evaluated by the HOST's powf, so the result
     * equals Texture.cpp:128-131 bit for bit), lut[256 + c] = c / 255 for alpha (:145-150).  The device expands them
     * into the float4 atlas: 3-4 bytes per texel cross PCIe instead of 16. */
    const uint8_t* texels8;
    int32_t channels;
    const float* lut;
} rt_texture;

typedef struct rt_mesh {
    const rt_bvh_node* nodes; int32_t num_nodes;
    const rt_tri* tris;       int32_t num_tris;
    const rt_shade* shade;    /* num_tris entries */
    const rt_texture* textures; int32_t num_textures;
} rt_mesh;

typedef struct rt_light {   /* LightData, Src/Light.h:16-21 */
    int32_t type;
    float pos_or_dir[3];
    float color[3];
} rt_light;

typedef struct rt_scene_desc {
    uint32_t abi_version;   /* RT_GPU_ABI_VERSION */
    const rt_shape* shapes;       int32_t num_shapes;     /* insertion order = test order */
    const rt_material* materials; int32_t num_materials;
    const rt_mesh* meshes;        int32_t num_meshes;
    const rt_light* lights;       int32_t num_lights;
    /* PseudoRandomUnitVectors (Math.cpp:17-31): xyz triples; needed by Diffuse materials. */
    const float* unit_vectors;    uint32_t num_unit_vectors;
    float eye[3];           /* ViewPoint, RayTracerProgram.cpp:133 = (0,0,7) */
    float dir_z;            /* RayTracerProgram.cpp:164 = -0.5 */
    float ray_distance;     /* RayTracerProgram.cpp:165 = 1000 */
    float bounce_offset;    /* BounceRayStartOffset, SurfaceMaterials.cpp:13 = 1e-4 */
} rt_scene_desc;

/* ---- render task ------------------------------------------------------------------------ */

enum {
    RT_MODE_PATH = 0,       /* RayTracerScene::RayTrace, RenderOption.UseBaseColor=false */
    RT_MODE_PREVIEW = 1,    /* RenderOption.UseBaseColor=true (RayTracerScene.cpp:54-61) */
    RT_MODE_WHITTED = 2,    /* primary hit + CalculateLightColor per light (RayTracerScene.cpp:127-175) */
    RT_MODE_PRIMARY = 3,    /* nearest hit only: ids + distance, no shading */
    RT_MODE_GUIDES = 4      /* RT_MODE_PRIMARY plus the HitNormal of the nearest hit, the guides of rt_gpu_denoise: one
                               un-jittered camera ray per pixel (antialias and pass_count are ignored), ids and distance
                               written exactly as RT_MODE_PRIMARY writes them, and {HitNormal.xyz, 0} (zeros on a miss)
                               into the frame slot's guide buffer (RT_READ_GUIDE_NORMAL_F32).  The buffer is allocated
                               (zeroed) by the slot's first GUIDES call and reallocated with the frame; accuBuffer,
                               bitcolor, the preview colour and the moments are left alone. */
};

enum {
    RT_TRAVERSE_EXACT = 0,  /* visit exactly the nodes the reference visits */
    RT_TRAVERSE_CULLED = 1  /* skip subtrees that cannot contain an accepted hit (same results) */
};

typedef struct rt_render_params {
    int32_t width, height;  /* replaces bitmapWidth/bitmapHeight (ColorBuffer.h:15-16) */
    int32_t start, end;     /* RenderThreadTask::Start / End (INCLUSIVE), pixel = y*width+x */
    int32_t mode;           /* RT_MODE_* */
    int32_t max_bounce;     /* MaxBounceTimes (RayTracerProgram.cpp:232); counts the primary segment */
    int32_t pass_begin;     /* first pass index (RNG key and ordering) */
    int32_t pass_count;     /* passes rendered by this call; each adds one AccumulatePixel sample */
    int32_t antialias;      /* 1: ENABLE_ANTIALIASING path, 4 jittered rays/pass (:146-169);
                               0: one un-jittered ray through (dx,dy,dir_z) per pass */
    uint32_t seed;          /* counter-RNG seed (include/rt_rng.h) */
    int32_t traverse;       /* RT_TRAVERSE_* */
    /* multi-GPU tile ownership: a pixel is rendered iff tile_count <= 1 or
     * ((y/tile_size)*ceil(width/tile_size) + x/tile_size) % tile_count == tile_rank */
    int32_t tile_size, tile_count, tile_rank;
} rt_render_params;

/* ---- readback ---------------------------------------------------------------------------- */

enum {
    RT_READ_ACCUM_RGBN_F32 = 0,   /* width*height x {sum.r,sum.g,sum.b,(float)Num}  (accuBuffer[]) */
    RT_READ_DISPLAY_ARGB8 = 1,    /* width*height x uint32 ARGB (bitcolor[]), gamma 2.2 (ColorBuffer.h:81-109) */
    RT_READ_PRIMARY_IDS_I32X2 = 2,/* width*height x {shape index, triangle index} of the primary hit, -1 = none */
    RT_READ_PRIMARY_DIST_F32 = 3, /* width*height x RayHitResult::Distance of the primary hit (0 if none) */
    RT_READ_COUNTERS_U64 = 4,     /* rt_counters */
    RT_READ_PREVIEW_RGBA_F32 = 5, /* width*height x float4: the linear colour c of the last RT_MODE_PREVIEW pass, the value the
                                     reference hands to LinearToGamma before it stores bitcolor (RayTracerProgram.cpp:175-180) */
    RT_READ_MOMENTS_F32 = 6,      /* width*height x float4 {M2.r, M2.g, M2.b, passes}: the moments of rt_gpu_track_moments
                                     (RT_ERR_NO_SCENE if tracking has never been on for the frame slot) */
    RT_READ_GUIDE_NORMAL_F32 = 7  /* width*height x float4 {HitNormal.xyz, 0} of the last RT_MODE_GUIDES render (RT_ERR_NO_SCENE
                                     if the frame slot has none) */
};

typedef struct rt_counters {
    uint64_t rays;          /* nearest-hit queries (FindIntersectionWithScene calls) + shadow queries */
    uint64_t camera_rays;
    uint64_t shadow_rays;
    uint64_t node_tests;    /* slab tests the reference algorithm evaluates (BVH nodes + shape bounds) */
    uint64_t tri_tests;     /* triangle tests the reference algorithm evaluates */
    uint64_t node_visits;   /* slab tests this implementation actually evaluated */
    uint64_t tri_visits;    /* triangle tests this implementation actually evaluated */
    uint64_t mesh_hits;     /* nearest-hit queries that ended on a mesh triangle (shading record fetched) */
    uint64_t mesh_walks;    /* KdTree::TestRayIntersection calls: queries that entered a mesh's bounds (MeshShape.cpp:284) */
} rt_counters;

typedef struct rt_gpu_ctx rt_gpu_ctx;

int rt_gpu_abi_version(void);
int rt_gpu_device_count(void);

/* Lifetime: one opaque context per GPU (replaces the process-wide singletons). */
int rt_gpu_create(int device, rt_gpu_ctx** out_ctx);
int rt_gpu_destroy(rt_gpu_ctx* ctx);
const char* rt_gpu_last_error(rt_gpu_ctx* ctx);   /* ctx may be NULL: last create() error */

/* Copies the whole scene to the device; the caller keeps ownership of all host memory and may
 * free it on return.  A second upload replaces the scene.  RT_ERR_INVALID (the context keeps its scene) for a
 * malformed description, a material graph it refuses (see rt_material), and a mesh with a non-finite (NaN or
 * infinite) BVH node bound or triangle corner p0 / p1 / p2; the message names the mesh.  The precomputed face normal
 * n is not checked: finite corners whose cross product overflows give a NaN n, and the reference computes the same. */
int rt_gpu_upload_scene(rt_gpu_ctx* ctx, const rt_scene_desc* scene);

/* Frame slots.  A context holds RT_GPU_FRAME_SLOTS independent sets of frame buffers (accuBuffer, bitcolor,
 * primary ids / distance), each with its own stream; rt_gpu_set_frame_slot chooses the set that the calls
 * after it address (reset_accum, render_tile, pack / unpack / push, resolve_display, readback, synchronize,
 * rt_gpu_stream, rt_gpu_accum_device_ptr, export_frame).  Within a slot calls execute in the order they were
 * made; calls on different slots are NOT ordered against each other on the device, so a driver can enqueue
 * frame k+1 on the other slot while the thin last bounce rounds, the exchange and the read-back of frame k
 * are still in flight (the reference's workers are never idle while tasks exist, ThreadTaskQueue.h:84-93; a
 * wavefront has a tail, and the next frame fills it).  Results do not depend on it.  Default slot: 0. */
#define RT_GPU_FRAME_SLOTS 4
int rt_gpu_set_frame_slot(rt_gpu_ctx* ctx, int32_t slot);
int rt_gpu_get_frame_slot(rt_gpu_ctx* ctx);
/* The frame size of the current frame slot (0 x 0 before its first reset_accum or render); either pointer may be NULL. */
int rt_gpu_frame_size(rt_gpu_ctx* ctx, int32_t* width, int32_t* height);

/* (Re)allocates width*height accumulation/display/primary buffers and zeroes them. */
int rt_gpu_reset_accum(rt_gpu_ctx* ctx, int32_t width, int32_t height);

/* Enqueues one render task on the context's stream and returns immediately.
 * If the buffers do not match params->width/height they are reset first. */
int rt_gpu_render_tile(rt_gpu_ctx* ctx, const rt_render_params* params);

/* ---- cameras -----------------------------------------------------------------------------------
 * A camera of one render call: the eye, the orientation and the image plane, in place of the uploaded scene's
 * eye / dir_z / ray_distance and the reference's fixed view down -z.  Nothing is kept: the next call without a
 * camera renders the uploaded view again. */
typedef struct rt_camera {
    float eye[3];          /* origin of every camera ray */
    float right[3];        /* world direction of camera-space +x (the reference's dx axis) */
    float up[3];           /* world direction of camera-space +y (dy) */
    float back[3];         /* world direction of camera-space +z: the camera looks along -back when dir_z < 0 */
    float dir_z;           /* camera-space z of the image plane (the reference's -0.5; sets the field of view) */
    float ray_distance;    /* Distance of camera rays (bounce segments are not affected) */
} rt_camera;

/* rt_gpu_render_tile with the camera rays of `camera`.  camera == NULL is exactly rt_gpu_render_tile(ctx, params);
 * every other rule of render_tile applies unchanged (frame slot, pass chunks, tiles, counters, last_render_ms,
 * kernel-class timing; enqueues and returns).
 * The camera ray of (pixel, sub-sample): v = (dx + ox, dy + oy, dir_z) with dx, dy, ox, oy and their rand() draws
 * those of render_tile (RayTracerProgram.cpp:133-165).  If right, up and back are exactly (1,0,0), (0,1,0), (0,0,1)
 * (compared as floats, so -0 is 0) the direction is normalized(v): the reference's generator with the camera's eye,
 * dir_z and distance.  Otherwise w[c] = (v.x*right[c] + v.y*up[c]) + v.z*back[c], in fp32, one rounding per
 * operation in that order, and the direction is normalized(w) (RVec3::GetNormalizedVec3: short vectors unchanged).
 * The basis need not be orthonormal; the image keeps the reference's mirroring in x.  Different frame slots may
 * render different cameras at the same time, and tiled ranks that pass the same camera assemble the same frame.
 * RT_ERR_INVALID, with nothing enqueued, for a non-finite field, a basis whose determinant (in double) is 0, and
 * every error of render_tile. */
int rt_gpu_render_view(rt_gpu_ctx* ctx, const rt_render_params* params, const rt_camera* camera);

/* ---- adaptive sampling -------------------------------------------------------------------------
 * accuBuffer keeps a sample count per pixel (RayTracerProgram.cpp:57-71), so pixels may hold different numbers of passes.
 * These calls let a driver spend passes where a pixel's error estimate is high.  A pixel's samples are keyed by
 * (seed, pixel, pass) (include/rt_rng.h), so a pixel that a masked call renders for passes [b, b + k) receives exactly
 * the samples a render_tile of those passes gives it.
 *
 * rt_gpu_track_moments: on != 0 turns tracking on for the current frame slot: it allocates a width*height float4 moment
 * buffer for the slot (the first time) and zeroes it, stream-ordered (every call with on != 0 zeroes it).  Without a
 * frame yet, the buffer comes with the frame.  While tracking is on, the fold of every RT_MODE_PATH and RT_MODE_WHITTED
 * render on the slot (render_tile, render_view, render_masked) also updates the buffer, per pixel and pass with the
 * pass colour x that the fold adds to sum (antialiased: the /4 average), channels r, g, b, in fp32 with one rounding per
 * operation in this order: n = Num before the pass, s0 the sum before and s1 = s0 + x the fold's own sum after it;
 * if n > 0, M2 += (x - s0 / (float)n) * (x - s1 / (float)(n + 1)); .w += 1 (the passes the moments cover).  PREVIEW and
 * PRIMARY leave it alone, as they leave accuBuffer.  rt_gpu_reset_accum zeroes it while tracking is on, a frame resize
 * reallocates it (zeroed), and it is read back with RT_READ_MOMENTS_F32.  on == 0 stops the updates and keeps the buffer.
 * With tracking off, renders run exactly the code they ran before. */
int rt_gpu_track_moments(rt_gpu_ctx* ctx, int32_t on);

/* render_tile (camera == NULL) or render_view (camera != NULL) restricted to a mask: a pixel is rendered iff it is inside
 * [start, end], owned under the tile fields, and mask[pixel] != 0.  `mask`: DEVICE memory of the context's GPU,
 * width*height bytes, read after everything enqueued on `stream` (a cudaStream_t; NULL = the current frame slot's stream)
 * before the call; work enqueued on `stream` after the call runs after the mask has been read (so the caller may free
 * or overwrite it in that stream's order), not after the render.  The work runs on the slot's stream like render_tile's, and every other rule of render_tile applies
 * unchanged: modes, passes, pass chunks, pipes, frame slot, counters (camera_rays counts the rendered pixels x passes x
 * rays per pass), last_render_ms and kernel-class timing, errors.  The pixels not rendered keep every frame buffer as it
 * was.  The mask is compacted on the device into a per-slot list of pixels in 8x4-block order (no host read), and the
 * grids stay those of the whole task.  RT_ERR_INVALID, with nothing enqueued, for a NULL mask, a mask that is not device
 * memory of the context's GPU, and every error of render_tile / render_view. */
int rt_gpu_render_masked(rt_gpu_ctx* ctx, const rt_render_params* params, const rt_camera* camera, const uint8_t* mask,
                         void* stream);

typedef struct rt_select_params {
    int32_t min_passes;     /* >= 2: pixels with fewer passes are selected */
    int32_t max_passes;     /* >= min_passes: pixels with this many passes or more are never selected */
    float abs_tol;          /* finite, >= 0 */
    float rel_tol;          /* finite, >= 0: tolerance relative to the pixel's mean luminance */
} rt_select_params;

/* The pixels of `region` (its frame size, which must equal the current frame slot's, [start, end] and tile fields) whose
 * error estimate calls for more passes.  With n = Num and m the slot's moments, mask[pixel] = 1 iff the pixel is in the
 * region, n < max_passes, and one of: n < min_passes; m.w != n (the moments do not cover every pass: error unknown);
 * se_c > abs_tol + rel_tol * Y for some channel c, where, in fp32 with one rounding per operation,
 * se_c = sqrtf((M2_c / (float)(n - 1)) / (float)n), Y = (0.2126f*mean_r + 0.7152f*mean_g) + 0.0722f*mean_b and
 * mean_c = sum_c / (float)n.  A comparison with NaN is false, so a NaN estimate or tolerance selects nothing.  Every other
 * pixel gets 0.  *count (DEVICE int32) = the number of ones.  `mask`: DEVICE, width*height bytes.  The inputs are read on
 * the slot's stream after its earlier work, and after everything enqueued on `stream` (NULL = the slot's stream) before
 * the call; the outputs are complete for work enqueued on `stream` after it.  RT_ERR_INVALID, with nothing enqueued, for
 * min_passes < 2 or max_passes < min_passes, a non-finite or negative tolerance, a slot on which tracking has never been
 * on, a region that does not match the frame (size, range, tile fields), and NULL, misaligned or non-device pointers. */
int rt_gpu_select_pixels(rt_gpu_ctx* ctx, const rt_render_params* region, const rt_select_params* s, uint8_t* mask,
                         int32_t* count, void* stream);

/* ---- denoising ------------------------------------------------------------------------------------
 * An edge-avoiding a-trous wavelet filter (Dammertz et al. 2010) of the current frame slot's mean colour, guided by the
 * first hit of an RT_MODE_GUIDES render (shape id, distance, normal), with a luminance weight driven by each pixel's
 * variance carried through the levels (the spatial part of SVGF).  Defined with + - * /, sqrtf and comparisons in fp32,
 * one rounding per operation, in the order written; Y(v) = (0.2126f*v.r + 0.7152f*v.g) + 0.0722f*v.b.
 *
 * Level 0, per pixel p, from acc = accuBuffer, m = the moments, a = the preview colour, the slot's primary ids (shape)
 * and distance (z) and the guide normal N:
 *   n = (int)acc.w; c = acc.rgb / (float)n; p is VALID iff n > 0 and acc.r, acc.g, acc.b are finite.
 *   use_albedo: d_ch = a_ch > 1e-3f ? a_ch : 1e-3f and x = c / d per channel; otherwise d = 1, x = c.
 *   use_variance, n >= 2 and m.w == (float)n: v = (Y(m.rgb) / (float)(n - 1)) / (float)n, then v = v / (Y(d) * Y(d)) with
 *   use_albedo; otherwise v = 0.
 * Level k = 0 .. levels-1, step s = 2^k.  An invalid p keeps x and v.  A valid p sums over the taps q = p + s*(i, j),
 * i, j in [-2, 2], j outer and i inner, skipping taps outside the frame, invalid taps and taps with shape_q != shape_p:
 *   centre tap (i = j = 0): w = 0.140625f;
 *   other taps: h = H[i+2] * H[j+2] with H = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
 *     if shape_p >= 0 (a hit): w_n = (N_p.x*N_q.x + N_p.y*N_q.y) + N_p.z*N_q.z, w_n = w_n > 0 ? w_n : 0, then
 *       w_n = w_n * w_n normal_log2 times; w_z = 1 / (1 + |z_p - z_q| / ((sigma_depth * (float)s) * z_p));
 *     a miss: w_n = w_z = 1;
 *     t = |Y(x_p) - Y(x_q)| / (sigma_lum * sqrtf(v_p) + lum_floor); w_l = 1 / (1 + t*t);
 *     w = ((h * w_n) * w_z) * w_l, and the tap is skipped unless w is finite;
 *   W += w; X += w * x_q (per channel); V += (w * w) * v_q;  then x = X / W, v = V / (W * W).
 * Output, per pixel: n <= 0 -> rgba = 0 and argb = 0; non-finite sums -> rgba = {c, (float)n} (the unfiltered mean);
 * otherwise rgba = {x * d, (float)n}.  argb (if given) = LinearToGamma + MakePixelColor of rgba.rgb, the display's
 * packing (0 for n <= 0, as bitcolor after rt_gpu_reset_accum).
 *
 * The guides are the slot's primary ids, distance and guide normal as last written; render RT_MODE_GUIDES over the
 * frame (a tiled multi-GPU driver: on the root, after the frame is assembled there) before denoising.  `rgba`: DEVICE,
 * width*height float4, 16-byte aligned; `argb`: DEVICE width*height uint32, or NULL.  The inputs are read on the slot's
 * stream after its earlier work, and after everything enqueued on `stream` (a cudaStream_t; NULL = the slot's stream)
 * before the call; the outputs are complete for work enqueued on `stream` after it.  No host read; no frame buffer of the
 * slot is written.  RT_ERR_INVALID, with nothing enqueued, for: a slot without a frame or without an RT_MODE_GUIDES
 * render since its frame was allocated; use_albedo without a preview pass on the slot; use_variance on a slot on which
 * tracking has never been on; a parameter out of range; NULL, misaligned or non-device pointers. */
typedef struct rt_denoise_params {
    int32_t levels;         /* 1..6 */
    int32_t use_albedo;     /* 0/1: demodulate by the slot's preview colour (RT_MODE_PREVIEW) */
    int32_t use_variance;   /* 0/1: the variance of each pixel's mean from the slot's moments (rt_gpu_track_moments) */
    int32_t normal_log2;    /* 0..8: the normal weight is the clamped dot product to the power 2^normal_log2 */
    float sigma_lum;        /* finite, >= 0 */
    float sigma_depth;      /* finite, > 0 */
    float lum_floor;        /* finite, > 0 */
} rt_denoise_params;

int rt_gpu_denoise(rt_gpu_ctx* ctx, const rt_denoise_params* p, float* rgba, uint32_t* argb, void* stream);

/* ---- ray queries on device memory -------------------------------------------------------------
 * Batches of the caller's own rays through the same wavefront kernels as render_tile (generate -> packet /
 * lane-per-walk / long walk -> shade, one round per mesh a ray reaches), results in device memory: picking,
 * visibility and shadow masks, cameras of one's own, bakes.  Results equal rt_gpu_trace_rays bit for bit. */
enum {
    RT_QUERY_NEAREST = 0,   /* RayTracerScene::FindIntersectionWithScene (RayTracerScene.cpp:99-125) */
    RT_QUERY_ANY = 1        /* the shadow loop of CalculateLightColor (:152-164): any accepted hit within Distance */
};

typedef struct rt_ray_query {
    const float* rays;      /* DEVICE, n x 7 floats {origin, direction, Distance}: the rays of rt_gpu_trace_rays */
    int32_t n;
    int32_t kind;           /* RT_QUERY_* */
    int32_t traverse;       /* RT_TRAVERSE_* (same results either way) */
    int32_t* shape;         /* DEVICE, n.  NEAREST: index of the shape hit, -1 = none;  ANY: 1 occluded, 0 not */
    int32_t* tri;           /* DEVICE, n, may be NULL; NEAREST only: original triangle id, -1 for analytic shapes / miss */
    float* hit;             /* DEVICE, n x 11, may be NULL; NEAREST only: HitPosition, HitNormal, Distance, SampledColor,
                               SampledAlpha, zeros on a miss (rt_gpu_trace_rays' hit11) */
} rt_ray_query;

/* Enqueues the queries on `stream` (a cudaStream_t; NULL = the current frame slot's stream) and returns at once:
 * the work is ordered after everything enqueued on `stream` before the call, and the outputs are complete for
 * everything enqueued on it after.  Every pointer must be device memory of the context's GPU.  n == 0 is a no-op.
 * Adds to the context's counters (rays; shadow_rays for RT_QUERY_ANY; slab / triangle tests, mesh walks and hits);
 * those are read on the context's stream, so order it after `stream` before reading them.  Leaves the frame
 * buffers, the frame slot and rt_gpu_last_render_ms alone. */
int rt_gpu_query_rays(rt_gpu_ctx* ctx, const rt_ray_query* q, void* stream);

/* Radiance of the caller's rays: what render_tile computes for one camera ray, started from ray i of the batch
 * instead — the path of RayTrace (RT_MODE_PATH), its UseBaseColor branch (RT_MODE_PREVIEW) or the Whitted composition
 * (RT_MODE_WHITTED).  Ray i draws rand() from the stream rt_rng_key(seed, stream_i, sample) (include/rt_rng.h),
 * starting at draw first_draw.  So render_tile's sample (pixel p, sample s) is reproduced bit for bit by its camera
 * ray with stream_i = p, sample = s and first_draw = 0 (un-jittered) or 2 (a jittered ray has drawn its two offsets). */
typedef struct rt_radiance_query {
    const float* rays;          /* DEVICE, n x 7 {origin, direction, Distance} (as rt_ray_query), 4-byte aligned */
    int32_t n;
    int32_t mode;               /* RT_MODE_PATH, RT_MODE_PREVIEW or RT_MODE_WHITTED */
    int32_t max_bounce;         /* MaxBounceTimes counting this segment, in [0, 32]; PATH/PREVIEW: 0 = black (RayTrace(ray, 0));
                                   WHITTED ignores it */
    int32_t traverse;           /* RT_TRAVERSE_* (same results either way) */
    uint32_t seed;              /* ray i draws rand() from rt_rng_key(seed, stream_i, sample), starting at draw first_draw */
    uint32_t sample;
    const uint32_t* rng_stream; /* DEVICE, n, may be NULL: stream_i = rng_stream_base + i */
    uint32_t rng_stream_base;
    uint32_t first_draw;        /* draws already consumed (2 = a jittered camera ray of render_tile) */
    float* rgba;                /* DEVICE, n x 4, 16-byte aligned: the radiance RayTrace / the Whitted composition returns, .w = 0 */
} rt_radiance_query;

/* Stream, ordering and pointer rules of rt_gpu_query_rays; n == 0 is a no-op.  Adds to the counters rays, shadow_rays
 * (Whitted light rays), slab / triangle tests, mesh walks and hits; camera_rays is not touched.  Leaves the frame
 * buffers, the frame slot and rt_gpu_last_render_ms alone.  RT_ERR_INVALID for another mode, max_bounce outside
 * [0, 32], (segments) x (mesh shapes) walks per path beyond the round table (as render_tile counts them), NULL or
 * misaligned rays / rgba, pointers that are not device memory of the context's GPU, and RT_MODE_PATH on a scene with
 * Diffuse materials but no unit-vector table. */
int rt_gpu_radiance_rays(rt_gpu_ctx* ctx, const rt_radiance_query* q, void* stream);

/* ---- scene updates on device memory ---------------------------------------------------------------
 * Geometry that moves (skinning, physics, a probe's surroundings) without a new rt_gpu_upload_scene.  After an
 * update, every later render, query and radiance call returns exactly what it would after a fresh upload of the same
 * scene with the mesh built by rt_host_add_mesh_arrays(points, point_idx, normals, normal_idx, ...) (the uploaded
 * texture coordinates and texture slot of each triangle stay), or with the shape records given.
 * Ordering: calls made on the context before an update see the old scene, calls made after it the new one, on any
 * frame slot and any stream, with no host synchronisation by the caller.  The update reads its inputs in `stream`'s
 * order (a cudaStream_t; NULL = the current frame slot's stream) and does not wait for frames in flight; it publishes
 * on the device once the calls enqueued before it have finished with the old scene, and later calls wait for that on
 * their streams.  Errors (RT_ERR_INVALID) leave the scene exactly as it was. */
typedef struct rt_mesh_update {
    const float* points;       /* DEVICE, num_points x 3, 4-byte aligned; every coordinate finite, the points no triangle
                                  uses too (they widen the shape's bounds); a NaN or infinity is refused */
    int32_t num_points;
    const int32_t* point_idx;  /* DEVICE, num_tris x 3: triangle t = original triangle id t */
    int32_t num_tris;          /* must equal the mesh's num_tris (as uploaded, or as the last rt_gpu_replace_mesh gave it) */
    const float* normals;      /* DEVICE, num_normals x 3, or NULL: every corner gets its triangle's cross(p1-p0, p2-p0) */
    int32_t num_normals;
    const int32_t* normal_idx; /* DEVICE, num_tris x 3, or NULL (exactly when normals is NULL) */
} rt_mesh_update;

/* New geometry for the mesh of mesh shape `shape`: the tree is rebuilt on the device (rt_gpu_build_bvh's rules), the
 * shading records, the shape's bounds (RAabb::Expand over all points) and the culling margin are recomputed.  The
 * builder reads one count per tree level on the host, so the call RETURNS ONCE THE BUILD IS COMPLETE: it waits for
 * `stream`'s earlier work and the build, not for renders on other streams.  The first update of a mesh allocates a
 * spare set of its arrays (192 B per triangle).  RT_ERR_INVALID for NULL, misaligned or non-device pointers, a shape
 * that is not a mesh or whose mesh another shape also references, num_tris other than the mesh's count, an
 * uploaded mesh whose node count is not 2 * num_tris - 1 (a description the host layer never produces),
 * num_points <= 0, normals without normal_idx or the reverse, and a point or normal index out of range or a non-finite
 * point coordinate (found on the device and read by the host before the build starts; nothing is published);
 * RT_ERR_NO_SCENE before an upload. */
int rt_gpu_update_mesh(rt_gpu_ctx* ctx, int32_t shape, const rt_mesh_update* u, void* stream);

/* A REFIT of the mesh of mesh shape `shape` to new points (per-frame deformation: skinning, cloth, physics): the
 * mesh's PUBLISHED tree (the uploaded one, or the one the last rt_gpu_update_mesh built) keeps its topology, that is
 * its node array, escapes, right-child words and leaf order; leaf slot j keeps triangle t = tris[j].index.  Recomputed:
 *   tris[j]      the record both builders emit for t from points[point_idx[3t+k]]: pads 0, n = cross(p1-p0, p2-p0),
 *                normalised (1.0f / sqrtf) iff |n|^2 >= FLT_EPSILON;
 *   leaf boxes   from FLT_MAX / -FLT_MAX, expanded with p0, p1, p2 in that order by < / >;
 *   inner boxes  the left child's box, a component taken from the right child's only where strictly smaller (min) or
 *                strictly larger (max): RAabb::Expand over the subtree's corners in leaf order.  This equals the
 *                builder's box in value, not always in the sign of a zero bound;
 *   shading records, the shape's bounds and the culling margin exactly as rt_gpu_update_mesh.
 * After a refit, every later call returns what a fresh upload of the scene with these arrays returns.  Ordering and
 * the spare set as rt_gpu_update_mesh, but the call RETURNS AT ONCE: no host read, no synchronisation, no blocking
 * allocation.  `status`: DEVICE int32 or NULL, written in `stream`'s order: 0 when the refit was published, otherwise
 * the bits of the device check (1 = a point index out of range, 2 = a normal index out of range, 16 = a non-finite
 * point coordinate, which the upload would refuse).  The mesh's arrays,
 * the shape's bounds and the culling margin are then left as they were, and every later call returns what it returned
 * before.  RT_ERR_INVALID (nothing enqueued) as rt_gpu_update_mesh's host-side checks, for a misaligned or non-device
 * `status`, and for an uploaded tree that is not a full binary tree over all its nodes whose leaves name every
 * triangle slot exactly once (the host layer always produces one; after an rt_gpu_update_mesh the builder's tree is
 * one); RT_ERR_NO_SCENE before an upload. */
int rt_gpu_refit_mesh(rt_gpu_ctx* ctx, int32_t shape, const rt_mesh_update* u, int32_t* status, void* stream);

/* A REPLACE of the mesh of mesh shape `shape`: new geometry of ANY triangle count, with its own texture coordinates and
 * texture slots (switching a level of detail, marching cubes or other geometry generated on the GPU, fracture,
 * streaming).  After a replace, every later call returns what a fresh upload returns of the scene in which the mesh is
 * rt_host_add_mesh_arrays(points, normals, texcoords, point_idx, normal_idx, texcoord_idx, num_tris) with
 * rt_shade.texture of triangle t = texture[t], the mesh keeps its uploaded rt_texture slots, and the shape's bounds are
 * RAabb::Expand over all the points.  Triangle ids that queries return are the new triangle order.  Ordering, blocking
 * (the call returns once the build is complete) as rt_gpu_update_mesh.  The uploaded mesh must
 * have at least one triangle; its node count and tree shape do not matter.  Afterwards the mesh is updatable and
 * refittable with the new count, and later updates and refits keep the new uv and slots.
 * Memory: the spare set is reused when it holds at least num_tris triangles, otherwise a set of num_tris is allocated
 * (stream-ordered on `stream`) and a spare set an earlier update allocated is released; capacity only grows.
 * RT_ERR_INVALID (the scene left exactly as it was) for rt_gpu_update_mesh's host-side checks other than the count and
 * node-count tests, num_tris <= 0, texcoords without texcoord_idx or the reverse, num_texcoords <= 0 with texcoords,
 * misaligned or non-device texcoords / texcoord_idx / texture, and, found on the device before anything is published, a
 * point, normal or texcoord index out of range, a texture slot the upload would refuse (>= the mesh's texture count,
 * or a slot without pixels; negative slots are untextured and pass) or a non-finite point coordinate; RT_ERR_NO_SCENE
 * before an upload. */
typedef struct rt_mesh_replace {
    rt_mesh_update geometry;      /* rt_mesh_update's rules, except that num_tris is the NEW triangle count (>= 1) */
    const float* texcoords;       /* DEVICE, num_texcoords x 2 {u, v}, 4-byte aligned, or NULL: every corner gets uv (0, 0) */
    int32_t num_texcoords;
    const int32_t* texcoord_idx;  /* DEVICE, num_tris x 3, or NULL (exactly when texcoords is NULL) */
    const int32_t* texture;       /* DEVICE, num_tris, or NULL (-1 everywhere): rt_shade.texture of triangle t, a slot of
                                     the mesh's UPLOADED textures */
} rt_mesh_replace;

int rt_gpu_replace_mesh(rt_gpu_ctx* ctx, int32_t shape, const rt_mesh_replace* r, void* stream);

/* Copies `count` caller records (host memory, consumed before return) over shapes [first, first + count): moved
 * spheres, planes, capsules and triangles, other materials.  type, mesh and has_bounds must equal the uploaded
 * record's and material must be in range (RT_ERR_INVALID otherwise); of a mesh record only `material` is taken (its
 * bounds are those of the mesh's current geometry).  Ordering as rt_gpu_update_mesh.  The records travel as kernel
 * parameters, so the call returns at once: it never waits on the host for frames in flight. */
int rt_gpu_update_shapes(rt_gpu_ctx* ctx, const rt_shape* shapes, int32_t first, int32_t count, void* stream);

/* Appearance updates: material nodes, lights and texels, for material editors, light placement, video or painted
 * textures and bakes that write back into a texture.  Ordering as rt_gpu_update_shapes: calls made before see the old
 * appearance, calls made after the new one, on any frame slot and stream, with no host synchronisation; the call
 * returns at once (no host wait, no blocking allocation).  Every error is found on the host: RT_ERR_INVALID with nothing
 * enqueued and the scene exactly as it was, RT_ERR_NO_SCENE before an upload.  After any sequence of them every later
 * call returns what a fresh rt_gpu_upload_scene of the edited description returns.
 *
 * rt_gpu_update_materials copies `count` caller records (host memory, consumed before return) over material nodes
 * [first, first + count).  first <= the current node count; a range past its end APPENDS nodes (the count only grows).
 * The graph as it will be afterwards must pass the upload's checks (type, children in range, no cycle, at most 8 Combine
 * nodes on any path from any node), so an update that closes a cycle through nodes it does not touch is refused.  A
 * Diffuse or Checker node on a scene without unit vectors makes later RT_MODE_PATH calls refuse, as after such an
 * upload; the update itself succeeds.  rt_gpu_update_shapes takes material indices below the new count. */
int rt_gpu_update_materials(rt_gpu_ctx* ctx, const rt_material* materials, int32_t first, int32_t count, void* stream);

/* Replaces the whole light list with `count` >= 0 caller records (host memory, consumed before return); the count may
 * differ from the uploaded one.  Later RT_MODE_WHITTED calls size their rounds (1 + lights) by the new count. */
int rt_gpu_update_lights(rt_gpu_ctx* ctx, const rt_light* lights, int32_t count, void* stream);

/* A rectangle of texels of one uploaded texture slot, from device memory.  Texel (x + i, y + j) of the slot becomes
 * rgba[j][i], or {lut[r], lut[g], lut[b], channels == 4 ? lut[256 + a] : 1.0f} of the 8-bit texel (what the upload
 * expands; rt_host_texel_lut gives the loader's table).  Slot sizes and atlas places do not change. */
typedef struct rt_texture_update {
    int32_t x, y, width, height;  /* rectangle of the slot's texels to overwrite, inside its uploaded size */
    const float* rgba;            /* DEVICE, `height` rows of width x {r,g,b,a} linear floats, `pitch` bytes apart; or NULL */
    size_t pitch;                 /* >= width * 16 */
    const uint8_t* texels8;       /* DEVICE, height x width x channels bytes, tightly packed; or NULL (exactly one of the two) */
    int32_t channels;             /* 3 or 4 with texels8 */
    const float* lut;             /* DEVICE, 512 floats with texels8: rt_texture's table */
} rt_texture_update;

/* Texture `slot` of mesh `mesh`.  width or height 0 is a no-op after the checks.  RT_ERR_INVALID for an unknown mesh or
 * slot, a slot that had no pixels at upload, a rectangle outside the slot, both or neither of rgba / texels8, channels
 * other than 3 or 4 with texels8, a pitch below width * 16 or not a multiple of 4, rgba or lut not 4-byte aligned, and a
 * source or lut that is not device memory of the context's GPU. */
int rt_gpu_update_texture(rt_gpu_ctx* ctx, int32_t mesh, int32_t slot, const rt_texture_update* t, void* stream);

/* Synchronises the stream, then copies `what` into caller memory (size-checked). */
int rt_gpu_readback(rt_gpu_ctx* ctx, int what, void* dst, size_t bytes);
int rt_gpu_synchronize(rt_gpu_ctx* ctx);

/* Device time (ms, CUDA events on the context's stream) of the most recent render_tile
 * kernel sequence; synchronises. */
int rt_gpu_last_render_ms(rt_gpu_ctx* ctx, float* out_ms);
/* Device time (ms) spent in the mesh-walk kernels (packet walk + lane-per-walk kernel; one timed bracket per
 * round per pass chunk) during the most recent render_tile made with rt_gpu_time_kernels(ctx, 1), summed, and
 * the number of brackets; synchronises.  Meaningful with one pipe (rt_gpu_set_pipes(ctx, 1)). */
int rt_gpu_last_kernel_ms(rt_gpu_ctx* ctx, float* out_ms, int32_t* out_launches);
int rt_gpu_reset_counters(rt_gpu_ctx* ctx);

/* Multi-GPU framebuffer exchange (the one exchange step of the path, SURVEY §8e).
 * pack:   gathers the pixels of the tiles this rank owns (per `params` tile fields) from the
 *         accumulation buffer into a dense device buffer of rt_gpu_owned_pixels() float4s.
 * unpack: scatters a peer's dense buffer back into this context's full-frame accumulation
 *         buffer.  `dev_ptr` is DEVICE memory on this context's GPU (e.g. a torch tensor that
 *         NCCL gathered into); the copy kernels run on the context's stream. */
int64_t rt_gpu_owned_pixels(int32_t width, int32_t height, int32_t tile_size,
                            int32_t tile_count, int32_t tile_rank);
int rt_gpu_pack_owned(rt_gpu_ctx* ctx, const rt_render_params* params, void* dev_ptr, size_t bytes);
int rt_gpu_unpack_owned(rt_gpu_ctx* ctx, const rt_render_params* params, int32_t src_rank,
                        const void* dev_ptr, size_t bytes);
/* Peer-memory variant (one process per GPU, GPUs that reach each other over NVLink / NVSwitch): the
 * root exports its accumulation buffer as a 64-byte CUDA IPC handle (after rt_gpu_reset_accum has
 * sized it; the buffer keeps its address while the frame size does not change), every other rank
 * opens it once and, after its passes, writes the tiles it owns straight into the root's frame —
 * no dense staging buffer and no collective.  The caller orders the ranks (any barrier on the
 * contexts' streams): root reset before the first push, all pushes before the root reads.
 * In ONE process driving several GPUs `peer_frame` may simply be rt_gpu_accum_device_ptr(root)
 * once peer access is enabled. */
int rt_gpu_export_frame(rt_gpu_ctx* ctx, void* handle64, size_t bytes);
int rt_gpu_open_peer_frame(rt_gpu_ctx* ctx, const void* handle64, size_t bytes, void** out_dev_ptr);
int rt_gpu_close_peer_frame(rt_gpu_ctx* ctx, void* dev_ptr);
int rt_gpu_push_owned(rt_gpu_ctx* ctx, const rt_render_params* params, void* peer_frame);
/* Delivery to HOST frames, every rank over its own PCIe link.  rt_gpu_register_host_frame pins and maps caller
 * memory into this context's GPU (cudaHostRegister, portable + mapped) — typically one POSIX shared-memory
 * frame that all ranks' processes hold — and returns its device address; rt_gpu_deliver_owned then writes the
 * tiles this rank owns (per `params`) from accuBuffer (16 B / pixel) and bitcolor (4 B / pixel) straight into
 * those frames (either may be NULL) on the slot's stream: the frame is assembled in host memory by N parallel
 * writers instead of being funnelled through the root GPU's one link.  The caller orders the ranks before it
 * reads (any barrier after each rank's stream has drained).  With tile_count <= 1 the whole frame is copied.
 * These are `bitcolor[]` / `accuBuffer[]` of RayTracerProgram.cpp:49,77 as the host sees them. */
int rt_gpu_register_host_frame(rt_gpu_ctx* ctx, void* host, size_t bytes, void** out_dev_ptr);
int rt_gpu_unregister_host_frame(rt_gpu_ctx* ctx, void* host);
int rt_gpu_deliver_owned(rt_gpu_ctx* ctx, const rt_render_params* params, void* host_accum_dev, void* host_display_dev);
/* Writes `value` into one 32-bit word of a registered host frame (its device address), ordered on the slot's
 * stream after everything enqueued before — e.g. "rank r has delivered frame k".  The consumer polls the words in
 * host memory: ranks need no collective, and none of them waits for another. */
int rt_gpu_signal_host(rt_gpu_ctx* ctx, void* host_word_dev, uint32_t value);
/* Single-process variant: gather every context's owned tiles into ctxs[root] with
 * cudaMemcpyPeerAsync (one host thread driving n GPUs). */
int rt_gpu_gather(rt_gpu_ctx** ctxs, int n, int root, const rt_render_params* params);

/* Recompute bitcolor[] = MakePixelColor(LinearToGamma(sum/Num)) from the accumulation buffer
 * (RayTracerProgram.cpp:68-71,185) — done automatically by render_tile for rendered pixels. */
int rt_gpu_resolve_display(rt_gpu_ctx* ctx);

/* The CUDA stream of the context as a cudaStream_t cast to void* (for event timing by callers). */
void* rt_gpu_stream(rt_gpu_ctx* ctx);
/* Device address of the full-frame accumulation buffer (width*height float4 {sum.rgb, Num}). */
void* rt_gpu_accum_device_ptr(rt_gpu_ctx* ctx);
/* Kernels this context has launched so far / device bytes held by the uploaded scene. */
uint64_t rt_gpu_launch_count(rt_gpu_ctx* ctx);
uint64_t rt_gpu_scene_bytes(rt_gpu_ctx* ctx);
/* Scheduling knobs (results never depend on them): queue entries a warp of the walk kernel pops at
 * once (multiple of 32); the number of walking lanes below which a warp stops to pop new entries;
 * how few lanes may still be looking for a leaf before the held leaves are tested; and the size of
 * a path pool in Ki records (0 = keep; a pool that fills up costs retry passes, never results). */
int rt_gpu_set_tuning(rt_gpu_ctx* ctx, int32_t window_items, int32_t min_lanes, int32_t leaf_wait,
                      int32_t pool_kpaths);
/* Pass chunks of a call are rendered by up to `pipes` concurrent streams (1 = strictly one kernel at a
 * time, which is what per-kernel event timing wants; default 4).  Results never depend on it. */
int rt_gpu_set_pipes(rt_gpu_ctx* ctx, int32_t pipes);     /* 0 restores the default */
int rt_gpu_get_pipes(rt_gpu_ctx* ctx);
/* Record a CUDA event pair around every walk-kernel launch so that rt_gpu_last_kernel_ms can report the
 * kernel's own time (off by default: ~20 extra stream operations per pass chunk). */
int rt_gpu_time_kernels(rt_gpu_ctx* ctx, int32_t on);
/* on = 2: instead, one event before EVERY launch of a render call, tagged with the kernel's class; afterwards
 * rt_gpu_kernel_class_ms reports, per class, the summed time from each launch's event to the next one and the
 * number of launches (use one pipe: the launches of a call then follow each other on one stream, so the
 * intervals are the kernels' durations plus launch gaps).  bench.py's roofline figures come from here. */
enum {
    RT_KERNEL_GENERATE = 0,     /* rt_generate_kernel */
    RT_KERNEL_PACKET_WALK = 1,  /* rt_walk_packet_kernel (round 0) */
    RT_KERNEL_WALK = 2,         /* rt_walk_kernel (bounce / shadow rounds; walks handed back by the packets) */
    RT_KERNEL_LONG_WALK = 3,    /* rt_longwalk_kernel */
    RT_KERNEL_SHADE = 4,        /* rt_shade_kernel */
    RT_KERNEL_FOLD = 5,         /* rt_resolve_kernel */
    RT_KERNEL_OTHER = 6,        /* memsets */
    RT_KERNEL_CLASSES = 7
};
int rt_gpu_kernel_class_ms(rt_gpu_ctx* ctx, float* ms, int32_t* launches, int32_t num_classes);

/* ---- mesh build on the device (SURVEY.md 8f-1) -------------------------------------------------
 * KdTree::Build (KdTree.cpp:10-126, 202-220) with the reference's partition rule, emitting the same
 * pre-order rt_bvh_node / leaf-order rt_tri arrays as the host builder, bit for bit.  `points` are xyz
 * triples, `indices` three point indices per triangle (host pointers); out_nodes holds 2*num_tris-1
 * records, out_tris num_tris.  out_depth / out_ms (device time of the build, CUDA events) may be NULL.
 * RT_ERR_INVALID for a point index out of range and for a non-finite (NaN or infinite) coordinate of any point,
 * which the upload would refuse too. */
int rt_gpu_build_bvh(rt_gpu_ctx* ctx, const float* points, int32_t num_points, const int32_t* indices,
                     int32_t num_tris, rt_bvh_node* out_nodes, rt_tri* out_tris, int32_t* out_depth, float* out_ms);

/* ---- verification hooks (used by tests/; same device code as the render path) ---------------
 * rt_gpu_trace_rays: n arbitrary rays {origin, direction, distance} (7 floats each) through the
 *   nearest-hit query that replaces RayTracerScene::FindIntersectionWithScene
 *   (RayTracerScene.cpp:99-125); hit11 = HitPosition, HitNormal, Distance, SampledColor,
 *   SampledAlpha per ray (zeros on a miss).  Host pointers.
 * rt_gpu_kat: primitive known-answer tests, one ray + one primitive per element.
 *   kind 0 RRay::TestIntersectionWithAabb (RRay.cpp:89-136; prim = min,max; out7[0] = tmin),
 *        1 ...WithTriangle (RRay.cpp:138-213; prim = p0,p1,p2), 2 ...WithSphere (RRay.cpp:25-64;
 *        prim = centre,radius), 3 ...WithPlane (RRay.cpp:66-87; prim = normal,point),
 *        4 RCapsule::TestRayIntersection (Shapes.cpp:34-125; prim = start,end,radius),
 *        5 Math::Q_rsqrt (MathHelper.cpp:26-38; prim = x; out7[0]),
 *        6 RMath::Barycentric (Math.cpp:56-68; prim = p,a,b,c; out7[0..2] = u,v,w),
 *        7 MakePixelColor(LinearToGamma(rgb)) (ColorBuffer.h:81-109; prim = rgb; flags = ARGB).
 *   flags[i] = accepted; out7 = HitPosition, HitNormal, Distance.  `rays` may be NULL for 5-7.
 * rt_gpu_kat_texture: RTexture::Sample (Texture.cpp:23-57) on the k-th texture of the uploaded
 *   scene (meshes in order, textured slots in order). */
int rt_gpu_trace_rays(rt_gpu_ctx* ctx, const float* rays, int32_t n, int32_t traverse,
                      int32_t* shape, int32_t* tri, float* hit11);
int rt_gpu_kat(rt_gpu_ctx* ctx, int32_t kind, const float* rays, const float* prims,
               int32_t prim_floats, int32_t n, int32_t* flags, float* out7);
int rt_gpu_kat_texture(rt_gpu_ctx* ctx, int32_t texture, const float* uv, int32_t n, float* out4);

#ifdef __cplusplus
}
#endif
#endif /* RT_GPU_H */
