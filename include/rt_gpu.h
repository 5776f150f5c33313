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
 *   rt_gpu_readback      replaces reading bitcolor[] / accuBuffer[] (:49,:77)
 *   rt_gpu_query_rays    FindIntersectionWithScene (RayTracerScene.cpp:99-125) and the shadow query of
 *                        CalculateLightColor (:152-164) on batches of the caller's rays in device memory
 *   rt_gpu_radiance_rays RayTracerScene::RayTrace (RayTracerScene.cpp:31-97), its preview branch, or the Whitted
 *                        composition, on batches of the caller's rays in device memory (own cameras, probes, bakes)
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

/* One node of a material tree (Blend/Combine reference children by index). */
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
    RT_MODE_PRIMARY = 3     /* nearest hit only: ids + distance, no shading */
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
    RT_READ_PREVIEW_RGBA_F32 = 5  /* width*height x float4: the linear colour c of the last RT_MODE_PREVIEW pass, the value the
                                     reference hands to LinearToGamma before it stores bitcolor (RayTracerProgram.cpp:175-180) */
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
 * free it on return.  A second upload replaces the scene. */
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

/* (Re)allocates width*height accumulation/display/primary buffers and zeroes them. */
int rt_gpu_reset_accum(rt_gpu_ctx* ctx, int32_t width, int32_t height);

/* Enqueues one render task on the context's stream and returns immediately.
 * If the buffers do not match params->width/height they are reset first. */
int rt_gpu_render_tile(rt_gpu_ctx* ctx, const rt_render_params* params);

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
    RT_KERNEL_OTHER = 6,        /* memsets, rt_finish_kernel */
    RT_KERNEL_CLASSES = 7
};
int rt_gpu_kernel_class_ms(rt_gpu_ctx* ctx, float* ms, int32_t* launches, int32_t num_classes);

/* ---- mesh build on the device (SURVEY.md 8f-1) -------------------------------------------------
 * KdTree::Build (KdTree.cpp:10-126, 202-220) with the reference's partition rule, emitting the same
 * pre-order rt_bvh_node / leaf-order rt_tri arrays as the host builder, bit for bit.  `points` are xyz
 * triples, `indices` three point indices per triangle (host pointers); out_nodes holds 2*num_tris-1
 * records, out_tris num_tris.  out_depth / out_ms (device time of the build, CUDA events) may be NULL. */
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
