// rt_scene_edit.cu — the scene edits behind include/rt_gpu.h: mesh updates, refits and replacements (a tree or boxes
// built on the device into a mesh's spare arrays, then published) and shape, material, light and texture updates.  An
// edit is enqueued on the caller's stream after every scene reader enqueued before it, and records the event every
// later reader waits for (wait_scene).  Lifetime, upload, render, queries and readback are rt_gpu.cu's.
//
// The whole file is compiled with -fmad=false, as rt_gpu.cu: device-built records match the host builder's bit for bit.
#include "rt_context.hpp"
#include "rt_bvh_core.hpp"

// kernels an upload launches too: defined in rt_gpu.cu (rt_patch_right_child in rt_wave_kernels.cuh, which only it includes)
__global__ void rt_expand_texels_kernel(cudaSurfaceObject_t atlas, const uint8_t* __restrict__ texels, const float* __restrict__ lut,
                                        int width, int height, int channels, int x0, int y0);
__global__ void rt_shade_leaf_order_kernel(const float4* __restrict__ tris, const float4* __restrict__ shade, float4* __restrict__ out, int n);
__global__ void rt_patch_right_child(rt_bvh_node* nodes, int n);

// ---- mesh updates, refits and replacements (rt_gpu_update_mesh, rt_gpu_refit_mesh, rt_gpu_replace_mesh) ----
// Bit flags of the index check (the builder's scratch flag for an update or a replace)
#define RT_UPD_BAD_POINT_INDEX 1
#define RT_UPD_BAD_NORMAL_INDEX 2
#define RT_UPD_BAD_TEXCOORD_INDEX 4
#define RT_UPD_BAD_TEXTURE 8
#define RT_UPD_BAD_POINT_VALUE 16

// Checks every index the call gives and copies the point indices into `safe_p`, the texcoord indices into `safe_t` and,
// when `safe_n` is given, the normal indices into it, with bad ones replaced by 0: no later kernel reads outside
// `points`, `normals` or `texcoords` even before the host has seen the flag.  (An update and a replace read normal_idx
// only once the host has seen it; a refit never waits for it, and throws its result away on the device.)  A replace
// also gives one texture slot per triangle: one the upload would refuse (>= the mesh's slot count, or a slot without
// pixels) is bad; negative slots pass.  Every point in [0, num_points) must be finite, the ones no triangle uses too:
// the shape's bounds are RAabb::Expand over all of them, and the upload refuses non-finite geometry for the walks'
// sake (rt_gpu_upload_scene).  Thread i checks index i (i < n) and point i (i < num_points).
__global__ void rt_update_check_kernel(const int* __restrict__ pidx, const float* __restrict__ points, int num_points,
                                       const int* __restrict__ nidx, int num_normals, const int* __restrict__ tidx, int num_texcoords,
                                       const int* __restrict__ texture, const DevMesh* __restrict__ mesh, int n,
                                       int* __restrict__ safe_p, int* __restrict__ safe_n, int* __restrict__ safe_t,
                                       int* __restrict__ flag)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < num_points)
    {
        const float* p = points + 3 * (size_t)i;
        if (!(fabsf(p[0]) <= FLT_MAX && fabsf(p[1]) <= FLT_MAX && fabsf(p[2]) <= FLT_MAX)) atomicOr(flag, RT_UPD_BAD_POINT_VALUE);
    }
    if (i >= n) return;
    int v = pidx[i], bad = 0;
    if (v < 0 || v >= num_points) { v = 0; bad |= RT_UPD_BAD_POINT_INDEX; }
    safe_p[i] = v;
    if (nidx)
    {
        int w = nidx[i];
        if (w < 0 || w >= num_normals) { w = 0; bad |= RT_UPD_BAD_NORMAL_INDEX; }
        if (safe_n) safe_n[i] = w;
    }
    if (tidx)
    {
        int w = tidx[i];
        if (w < 0 || w >= num_texcoords) { w = 0; bad |= RT_UPD_BAD_TEXCOORD_INDEX; }
        safe_t[i] = w;
    }
    if (texture && i % 3 == 0)
    {
        const int slot = texture[i / 3];
        if (slot >= mesh->num_textures || (slot >= 0 && mesh->textures[slot].width == 0)) bad |= RT_UPD_BAD_TEXTURE;
    }
    if (bad) atomicOr(flag, bad);
}

// The corner normals of triangle t into dst[0..8]: normals[nidx], or every corner the triangle's unnormalised geometric
// normal as host/mesh_loader.cpp computes it.
__device__ __forceinline__ void upd_corner_normals(float* dst, int t, const float* __restrict__ points, const int* __restrict__ pidx,
                                                   const float* __restrict__ normals, const int* __restrict__ nidx)
{
    if (normals)
        for (int k = 0; k < 3; k++)
        {
            const float* v = normals + 3 * (size_t)nidx[3 * (size_t)t + k];
            dst[3 * k] = v[0]; dst[3 * k + 1] = v[1]; dst[3 * k + 2] = v[2];
        }
    else
    {
        const float* p0 = points + 3 * (size_t)pidx[3 * (size_t)t];
        const float* p1 = points + 3 * (size_t)pidx[3 * (size_t)t + 1];
        const float* p2 = points + 3 * (size_t)pidx[3 * (size_t)t + 2];
        const float ax = p1[0] - p0[0], ay = p1[1] - p0[1], az = p1[2] - p0[2];
        const float bx = p2[0] - p0[0], by = p2[1] - p0[1], bz = p2[2] - p0[2];
        const float nx = rt_host_nan(ay * bz - az * by), ny = rt_host_nan(az * bx - ax * bz), nz = rt_host_nan(ax * by - ay * bx);
        for (int k = 0; k < 3; k++) { dst[3 * k] = nx; dst[3 * k + 1] = ny; dst[3 * k + 2] = nz; }
    }
}

// Shading records in ORIGINAL triangle order: the new normals, uv and texture slot from the published record.
// Published leaf record j belongs to triangle cur_tris[j].index.
__global__ void rt_update_shade_kernel(const float4* __restrict__ cur_tris, const float* __restrict__ cur_shade,
                                       const float* __restrict__ points, const int* __restrict__ pidx,
                                       const float* __restrict__ normals, const int* __restrict__ nidx, float* __restrict__ out, int n)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int t = __float_as_int(cur_tris[4 * (size_t)j].w);
    const float* src = cur_shade + 16 * (size_t)j;
    float* dst = out + 16 * (size_t)t;
    upd_corner_normals(dst, t, points, pidx, normals, nidx);
    for (int k = 9; k < 16; k++) dst[k] = src[k];           // uv0 uv1 uv2 texture
}

// A replace's shading records in original order: normals as rt_update_shade_kernel, uv copied from
// texcoords[tidx] (bits as given; (0, 0) without texcoords), the slot from `texture` (-1 without).
__global__ void rt_replace_shade_kernel(const float* __restrict__ points, const int* __restrict__ pidx,
                                        const float* __restrict__ normals, const int* __restrict__ nidx,
                                        const float* __restrict__ texcoords, const int* __restrict__ tidx,
                                        const int* __restrict__ texture, float* __restrict__ out, int n)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    float* dst = out + 16 * (size_t)t;
    upd_corner_normals(dst, t, points, pidx, normals, nidx);
    for (int k = 0; k < 3; k++)
    {
        float u = 0.0f, v = 0.0f;
        if (texcoords)
        {
            const float* uv = texcoords + 2 * (size_t)tidx[3 * (size_t)t + k];
            u = uv[0]; v = uv[1];
        }
        dst[9 + 2 * k] = u; dst[10 + 2 * k] = v;
    }
    dst[15] = __int_as_float(texture ? texture[t] : -1);
}

// RAabb::Expand over the points in array order as 64-bit keys: value order in the high word (-0 == +0, as `<`
// sees them), the point index in the low word so that ties go to the FIRST occurrence (min: index, max: ~index).
__device__ __forceinline__ unsigned upd_ord_bits(float v)
{
    unsigned b = __float_as_uint(v);
    if (v == 0.0f) b = 0u;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void rt_update_bounds_kernel(const float* __restrict__ points, int num_points, unsigned long long* keys)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long mn[3] = { ~0ull, ~0ull, ~0ull }, mx[3] = { 0ull, 0ull, 0ull };
    if (i < num_points)
        for (int c = 0; c < 3; c++)
        {
            const float v = points[3 * (size_t)i + c];
            if (v != v) continue;                                   // NaN never wins a < or > test
            const unsigned long long o = (unsigned long long)upd_ord_bits(v) << 32;
            mn[c] = o | (unsigned)i; mx[c] = o | (0xFFFFFFFFu - (unsigned)i);
        }
    for (int c = 0; c < 3; c++)
    {
        for (int o = 16; o > 0; o >>= 1)
        {
            const unsigned long long a = __shfl_xor_sync(0xffffffffu, mn[c], o), b = __shfl_xor_sync(0xffffffffu, mx[c], o);
            if (a < mn[c]) mn[c] = a;
            if (b > mx[c]) mx[c] = b;
        }
        if ((threadIdx.x & 31) == 0)
        {
            if (mn[c] != ~0ull) atomicMin(keys + c, mn[c]);
            if (mx[c] != 0ull) atomicMax(keys + 3 + c, mx[c]);
        }
    }
}

// The publication of a mesh edit (one thread, after the join): the mesh's record points at the new arrays of num_tris
// triangles and 2 * num_tris - 1 nodes, with the culling margin of the new root (as upload computes it); the shape gets
// the new bounds.  Kernels read both records at run time.  flag / status: a refit's (null otherwise).  With the flag
// set the arrays are a copy of the live set (rt_refit_restore_kernel), so the shape's bounds and the mesh's margin stay
// as they are; the flag goes to *status.
__global__ void rt_update_publish_kernel(DevMesh* meshes, int mesh, rt_shape* shapes, int shape, const rt_bvh_node* nodes,
                                         const rt_tri* tris, const rt_shade* shade, int num_tris, const unsigned long long* keys,
                                         const float* points, const int* flag, int* status)
{
    const int f = flag ? *flag : 0;
    if (status) *status = f;
    DevMesh& m = meshes[mesh];
    m.nodes = (const float4*)nodes; m.tris = (const float4*)tris; m.shade = (const float4*)shade;
    m.num_tris = num_tris; m.num_nodes = 2 * num_tris - 1;
    if (f) return;
    float scale = 0.0f;
    for (int k = 0; k < 3; k++)
    {
        scale = fmaxf(scale, fabsf(nodes[0].bmin[k]));
        scale = fmaxf(scale, fabsf(nodes[0].bmax[k]));
    }
    m.cull_scale = scale;
    rt_shape& s = shapes[shape];
    for (int c = 0; c < 3; c++)
    {
        float lo = FLT_MAX, hi = -FLT_MAX;                       // RAabb's empty box
        if (keys[c] != ~0ull)
        {
            const float v = points[3 * (size_t)(unsigned)(keys[c] & 0xFFFFFFFFull) + c];
            if (v < lo) lo = v;
        }
        if (keys[3 + c] != 0ull)
        {
            const float v = points[3 * (size_t)(0xFFFFFFFFu - (unsigned)(keys[3 + c] & 0xFFFFFFFFull)) + c];
            if (v > hi) hi = v;
        }
        s.bounds_min[c] = lo; s.bounds_max[c] = hi;
    }
}

// Parent links of the published tree (left child i+1, right child in the inner node's `tri` word, -2 - index; the root
// has none), the node of each leaf slot, and zeroed arrival counters.  rt_gpu_refit_mesh runs only on a full binary
// tree over all its nodes whose leaves name every slot once (MeshState::refittable), so every link is set and every
// node is reached by a climb.
__global__ void rt_refit_links_kernel(const rt_bvh_node* __restrict__ nodes, int n, int* __restrict__ parent,
                                      int* __restrict__ leaf_node, int* __restrict__ arrivals)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    arrivals[i] = 0;
    if (i == 0) parent[0] = -1;
    const int tri = nodes[i].tri;
    if (tri >= 0)
    {
        leaf_node[tri] = i;
        return;
    }
    parent[i + 1] = i;
    parent[-2 - tri] = i;
}

__device__ __forceinline__ void refit_store_node(float4* nodes, int i, const float* mn, int escape, const float* mx, int tri)
{
    nodes[2 * (size_t)i] = make_float4(mn[0], mn[1], mn[2], __int_as_float(escape));
    nodes[2 * (size_t)i + 1] = make_float4(mx[0], mx[1], mx[2], __int_as_float(tri));
}

// One thread per leaf slot j: the triangle record of t = cur_tris[j].index from the new corners and the leaf's box
// (RAabb's empty box expanded with p0, p1, p2 by < / >, as the host builder's loop over a one-triangle node), then
// up the tree: the SECOND child to arrive at an inner node combines both children's boxes, always left then right
// (a component of the right child's box only where strictly smaller / larger), so the result does not depend on which
// child finished first.  Escape and `tri` words are the published ones.
__global__ void rt_refit_kernel(const float4* __restrict__ cur_tris, const float4* __restrict__ cur_nodes,
                                const float* __restrict__ points, const int* __restrict__ pidx, const int* __restrict__ leaf_node,
                                const int* __restrict__ parent, int* arrivals, rt_tri* __restrict__ tris, float4* nodes, int T)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= T) return;
    const int t = __float_as_int(cur_tris[4 * (size_t)j].w);
    const rt_tri r = rt_tri_record(points + 3 * (size_t)pidx[3 * (size_t)t], points + 3 * (size_t)pidx[3 * (size_t)t + 1],
                                   points + 3 * (size_t)pidx[3 * (size_t)t + 2], t);
    tris[j] = r;
    int i = leaf_node[j];
    float mn[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, mx[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    const float* corner[3] = { r.p0, r.p1, r.p2 };
    for (int k = 0; k < 3; k++)
        for (int c = 0; c < 3; c++)
        {
            if (corner[k][c] < mn[c]) mn[c] = corner[k][c];
            if (corner[k][c] > mx[c]) mx[c] = corner[k][c];
        }
    float4 w0 = cur_nodes[2 * (size_t)i], w1 = cur_nodes[2 * (size_t)i + 1];
    refit_store_node(nodes, i, mn, __float_as_int(w0.w), mx, __float_as_int(w1.w));
    for (;;)
    {
        __threadfence();                                    // this node's box before the arrival that publishes it
        const int p = parent[i];
        if (p < 0) return;
        if (atomicAdd(arrivals + p, 1) == 0) return;        // the sibling is still on its way: it carries on
        __threadfence();
        w0 = cur_nodes[2 * (size_t)p]; w1 = cur_nodes[2 * (size_t)p + 1];
        const int right = -2 - __float_as_int(w1.w);
        const float4 l0 = __ldcg(nodes + 2 * (size_t)(p + 1)), l1 = __ldcg(nodes + 2 * (size_t)(p + 1) + 1);
        const float4 r0 = __ldcg(nodes + 2 * (size_t)right), r1 = __ldcg(nodes + 2 * (size_t)right + 1);
        mn[0] = l0.x; mn[1] = l0.y; mn[2] = l0.z; mx[0] = l1.x; mx[1] = l1.y; mx[2] = l1.z;
        if (r0.x < mn[0]) mn[0] = r0.x;
        if (r0.y < mn[1]) mn[1] = r0.y;
        if (r0.z < mn[2]) mn[2] = r0.z;
        if (r1.x > mx[0]) mx[0] = r1.x;
        if (r1.y > mx[1]) mx[1] = r1.y;
        if (r1.z > mx[2]) mx[2] = r1.z;
        refit_store_node(nodes, p, mn, __float_as_int(w0.w), mx, __float_as_int(w1.w));
        i = p;
    }
}

// A refit whose index check failed publishes an exact copy of the published set (the host's ping-pong swaps on
// every call, so the spare set must hold the live arrays afterwards); rt_update_publish_kernel then leaves the shape's
// bounds and the mesh's culling margin as they are.  Without the flag every block leaves at once.
__global__ void rt_refit_restore_kernel(const int* __restrict__ flag, const float4* __restrict__ cur_nodes,
                                        const float4* __restrict__ cur_tris, const float4* __restrict__ cur_shade, float4* nodes,
                                        float4* tris, float4* shade, int n, int T)
{
    if (*flag == 0) return;
    const size_t a = 2 * (size_t)n, b = 4 * (size_t)T;
    for (size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x; k < a + 2 * b; k += (size_t)gridDim.x * blockDim.x)
    {
        if (k < a) nodes[k] = cur_nodes[k];
        else if (k < a + b) tris[k - a] = cur_tris[k - a];
        else shade[k - a - b] = cur_shade[k - a - b];
    }
}

// rt_gpu_update_shapes: caller records over the device's; a mesh record gives its material only.  The records travel
// as the kernel's parameter (copied at launch: no staging buffer, nothing for the host to wait for).
#define RT_SHAPES_PER_LAUNCH 48                       // 48 x 80 B: within the classic 4 KB parameter space
struct ShapeBatch { rt_shape rec[RT_SHAPES_PER_LAUNCH]; };
__global__ void rt_update_shapes_kernel(rt_shape* shapes, ShapeBatch src, int count)
{
    const int k = threadIdx.x;
    if (k >= count) return;
    if (src.rec[k].type == RT_SHAPE_MESH) shapes[k].material = src.rec[k].material;
    else shapes[k] = src.rec[k];
}

// rt_gpu_update_materials / rt_gpu_update_lights: caller records travel the same way (28 B each)
#define RT_RECORDS_PER_LAUNCH 128                     // 128 x 28 B: within the classic 4 KB parameter space
template <typename T> struct RecordBatch { T rec[RT_RECORDS_PER_LAUNCH]; };
template <typename T>
__global__ void rt_update_records_kernel(T* dst, RecordBatch<T> src, int count)
{
    const int k = threadIdx.x;
    if (k < count) dst[k] = src.rec[k];
}

// Every stream of the context that runs scene readers (the frame slots' streams and the pipes, onto which render calls
// and queries fork) has finished what was enqueued on it before this call, in `st`'s order: the join of an update.
static int join_scene_readers(rt_gpu_ctx* ctx, cudaStream_t st)
{
    if (!ctx->join_event) RT_CUDA(cudaEventCreateWithFlags(&ctx->join_event, cudaEventDisableTiming));
    auto join = [&](cudaStream_t s) -> cudaError_t {
        if (!s || s == st) return cudaSuccess;
        cudaError_t e = cudaEventRecord(ctx->join_event, s);
        return e == cudaSuccess ? cudaStreamWaitEvent(st, ctx->join_event, 0) : e;
    };
    RT_CUDA(join(ctx->stream));
    for (int k = 0; k < RT_FRAME_SLOTS; k++)
        if (k != ctx->slot) RT_CUDA(join(ctx->parked[k].stream));
    for (int k = 0; k < RT_PIPES; k++) RT_CUDA(join(ctx->pipes[k].stream));
    return RT_OK;
}

static int publish_done(rt_gpu_ctx* ctx, cudaStream_t st)
{
    if (!ctx->scene_event) RT_CUDA(cudaEventCreateWithFlags(&ctx->scene_event, cudaEventDisableTiming));
    RT_CUDA(cudaEventRecord(ctx->scene_event, st));
    ctx->scene_event_live = true;
    return RT_OK;
}

// Stream-ordered device memory of the edits, and its release.  Scene arrays (`scene`: a mesh's spare set, grown material
// and light arrays) are listed in scene_allocs, which the next upload or destroy frees, and counted in scene_bytes; the
// update scratch belongs to the context and is neither.
static int alloc_pooled(rt_gpu_ctx* ctx, void** out, size_t bytes, cudaStream_t st, bool scene = true)
{
    *out = nullptr;
    RT_CUDA(cudaMallocAsync(out, bytes, st));
    if (scene)
    {
        ctx->scene_allocs.push_back(*out);
        ctx->scene_bytes += bytes;
    }
    return RT_OK;
}

static int free_pooled(rt_gpu_ctx* ctx, void* p, size_t bytes, cudaStream_t st, bool scene = true)
{
    RT_CUDA(cudaFreeAsync(p, st));
    if (scene)
    {
        ctx->scene_allocs.erase(std::find(ctx->scene_allocs.begin(), ctx->scene_allocs.end(), p));
        ctx->scene_bytes -= bytes;
    }
    return RT_OK;
}

// The host-side checks of rt_gpu_update_mesh, rt_gpu_refit_mesh and rt_gpu_replace_mesh (`fn` names the call in the
// messages); the shape's mesh goes to *mesh.  An update and a refit keep the published count (`same_count`); a replace
// takes any positive count and publishes a tree of its own, so the published node count does not matter to it.
static int check_mesh_update(rt_gpu_ctx* ctx, const char* fn, int32_t shape, const rt_mesh_update* u, bool same_count, int* mesh)
{
    const std::string f(fn);
    if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, f + " before rt_gpu_upload_scene");
    if (!u) return fail(ctx, RT_ERR_INVALID, f + ": update is null");
    if (shape < 0 || shape >= (int)ctx->host_shapes.size() || ctx->host_shapes[shape].type != RT_SHAPE_MESH)
        return fail(ctx, RT_ERR_INVALID, f + ": shape is not a mesh shape of the scene");
    const int mi = ctx->host_shapes[shape].mesh;
    const rt_gpu_ctx::MeshState& ms = ctx->mesh_state[mi];
    if (ms.users != 1) return fail(ctx, RT_ERR_INVALID, f + ": another shape references the same mesh");
    if (same_count)
    {
        if (ms.num_tris <= 0 || u->num_tris != ms.num_tris)
            return fail(ctx, RT_ERR_INVALID, f + ": num_tris differs from the uploaded mesh's");
        // the update publishes a tree of 2T-1 nodes in an array of that size; the walks read num_nodes as uploaded
        if (ms.num_nodes != 2 * ms.num_tris - 1)
            return fail(ctx, RT_ERR_INVALID, f + ": the uploaded mesh's node count is not 2 * num_tris - 1 (not a tree of its triangles)");
    }
    else
    {
        if (ms.num_tris <= 0) return fail(ctx, RT_ERR_INVALID, f + ": the uploaded mesh has no triangles");
        if (u->num_tris <= 0) return fail(ctx, RT_ERR_INVALID, f + ": num_tris must be positive");
    }
    if ((long long)u->num_tris * 3 >= 0xFFFFFFFFll) return fail(ctx, RT_ERR_INVALID, f + ": too many triangles");
    if (u->num_points <= 0) return fail(ctx, RT_ERR_INVALID, f + ": num_points must be positive");
    if (!u->points || !u->point_idx) return fail(ctx, RT_ERR_INVALID, f + ": points and point_idx are required");
    if ((u->normals == nullptr) != (u->normal_idx == nullptr))
        return fail(ctx, RT_ERR_INVALID, f + ": normals and normal_idx come together");
    if (u->normals && u->num_normals <= 0) return fail(ctx, RT_ERR_INVALID, f + ": num_normals must be positive");
    RT_CUDA(cudaSetDevice(ctx->device));
    const int rc = check_device_args(ctx, fn, { { u->points, "points", 4 }, { u->point_idx, "point_idx", 4 },
                                                { u->normals, "normals", 4 }, { u->normal_idx, "normal_idx", 4 } });
    if (rc != RT_OK) return rc;
    *mesh = mi;
    return RT_OK;
}

// A spare set of a mesh's arrays with room for `tris` triangles, on `st` after wait_scene: the spare set and the
// scratch were last read by work the previous update waited for, so a spare that is too small can be released here.
// Capacity only grows: a smaller count builds into the larger set.
static int alloc_spare(rt_gpu_ctx* ctx, rt_gpu_ctx::MeshState& ms, int tris, cudaStream_t st)
{
    if (ms.spare.nodes && ms.spare.cap >= tris) return RT_OK;
    int rc;
    if (ms.spare.pooled)
    {
        const size_t T = (size_t)ms.spare.cap;
        if ((rc = free_pooled(ctx, ms.spare.nodes, (2 * T - 1) * sizeof(rt_bvh_node), st)) != RT_OK) return rc;
        if ((rc = free_pooled(ctx, ms.spare.tris, T * sizeof(rt_tri), st)) != RT_OK) return rc;
        if ((rc = free_pooled(ctx, ms.spare.shade, T * sizeof(rt_shade), st)) != RT_OK) return rc;
    }
    ms.spare = rt_gpu_ctx::MeshArrays{ nullptr, nullptr, nullptr, 0, false };
    const size_t T = (size_t)tris;
    rt_gpu_ctx::MeshArrays a = { nullptr, nullptr, nullptr, tris, true };
    if ((rc = alloc_pooled(ctx, (void**)&a.nodes, (2 * T - 1) * sizeof(rt_bvh_node), st)) != RT_OK) return rc;
    if ((rc = alloc_pooled(ctx, (void**)&a.tris, T * sizeof(rt_tri), st)) != RT_OK) return rc;
    if ((rc = alloc_pooled(ctx, (void**)&a.shade, T * sizeof(rt_shade), st)) != RT_OK) return rc;
    ms.spare = a;
    return RT_OK;
}

// The update scratch as `layout` carves it: layout(Carve&) takes the call's arrays, once to size the block (which only
// grows) and once more on it.
template <typename Layout>
static int carve_update_scratch(rt_gpu_ctx* ctx, cudaStream_t st, Layout layout)
{
    Carve c = { nullptr, 0 };
    layout(c);
    if (c.off > ctx->update_scratch_cap)
    {
        int rc;
        if (ctx->update_scratch && (rc = free_pooled(ctx, ctx->update_scratch, 0, st, false)) != RT_OK) return rc;
        ctx->update_scratch = nullptr; ctx->update_scratch_cap = 0;
        if ((rc = alloc_pooled(ctx, &ctx->update_scratch, c.off, st, false)) != RT_OK) return rc;
        ctx->update_scratch_cap = c.off;
    }
    c = Carve{ (char*)ctx->update_scratch, 0 };
    layout(c);
    return RT_OK;
}

// The tail of every mesh edit, once the spare set holds the new tree and `shade_tmp` the shading records in original
// order: the records in leaf order, the bounds of u's points, then, once every call enqueued before this one has
// finished reading the old arrays, the publication of the spare set with T triangles and the swap.  flag / status: a
// refit's device check, which the host never reads, and the caller's status word (null for an update or a replace,
// whose check the host has seen): with the flag set the spare set gets a copy of the live one and the publication
// keeps the shape's bounds and the mesh's margin.
static int publish_mesh(rt_gpu_ctx* ctx, int32_t shape, int mi, int T, const rt_mesh_update* u, const rt_shade* shade_tmp,
                        unsigned long long* keys, const int* flag, int32_t* status, cudaStream_t st)
{
    rt_gpu_ctx::MeshState& ms = ctx->mesh_state[mi];
    rt_shade_leaf_order_kernel<<<(unsigned)((T + 255) / 256), 256, 0, st>>>((const float4*)ms.spare.tris, (const float4*)shade_tmp,
                                                                            (float4*)ms.spare.shade, T);
    RT_CUDA(cudaMemsetAsync(keys, 0xFF, 3 * sizeof(unsigned long long), st));
    RT_CUDA(cudaMemsetAsync(keys + 3, 0, 3 * sizeof(unsigned long long), st));
    rt_update_bounds_kernel<<<(unsigned)((u->num_points + 255) / 256), 256, 0, st>>>(u->points, u->num_points, keys);
    ctx->launches += 2;
    if (flag)
    {
        rt_refit_restore_kernel<<<(unsigned)ctx->num_sms * 4u, 256, 0, st>>>(
            flag, (const float4*)ms.cur.nodes, (const float4*)ms.cur.tris, (const float4*)ms.cur.shade, (float4*)ms.spare.nodes,
            (float4*)ms.spare.tris, (float4*)ms.spare.shade, 2 * T - 1, T);
        ctx->launches++;
    }
    RT_CUDA(cudaGetLastError());
    // publish once every call enqueued before this one has finished reading the old arrays
    int rc = join_scene_readers(ctx, st);
    if (rc != RT_OK) return rc;
    rt_update_publish_kernel<<<1, 1, 0, st>>>(const_cast<DevMesh*>(ctx->scene.meshes), mi, const_cast<rt_shape*>(ctx->scene.shapes),
                                              shape, ms.spare.nodes, ms.spare.tris, ms.spare.shade, T, keys, u->points, flag, status);
    RT_CUDA(cudaGetLastError());
    ctx->launches++;
    if ((rc = publish_done(ctx, st)) != RT_OK) return rc;
    std::swap(ms.cur, ms.spare);
    ms.num_tris = T; ms.num_nodes = 2 * T - 1;
    ms.refittable = true;                   // the builder's tree, or the refitted one
    return RT_OK;
}

// The body of rt_gpu_update_mesh and rt_gpu_replace_mesh after their host checks: the device check, a tree of
// r->geometry.num_tris triangles built into the spare set, the shading records (uv and slot from the published records
// for an update, from the caller's arrays for a `replace`), then publish_mesh.  Returns once the build is complete.
static int rebuild_mesh(rt_gpu_ctx* ctx, const char* fn, int32_t shape, int mi, const rt_mesh_replace* r, bool replace, cudaStream_t st)
{
    const rt_mesh_update* u = &r->geometry;
    rt_gpu_ctx::MeshState& ms = ctx->mesh_state[mi];
    const int T = u->num_tris;
    RT_CUDA(wait_scene(ctx, st));
    int rc;
    if ((rc = alloc_spare(ctx, ms, T, st)) != RT_OK) return rc;
    // scratch: the builder's block (its flag is the check's), safe point indices (3T), safe texcoord indices (3T, a
    // replace with texcoords only), shading records in original order (T), bounds keys (6)
    char* build; int *safe_idx, *safe_tidx; rt_shade* shade_tmp; unsigned long long* keys;
    rc = carve_update_scratch(ctx, st, [&](Carve& c) {
        build = c.take<char>(rt_bvh_scratch_bytes(T));
        safe_idx = c.take<int>(3 * (size_t)T);
        safe_tidx = r->texcoord_idx ? c.take<int>(3 * (size_t)T) : nullptr;
        shade_tmp = c.take<rt_shade>((size_t)T);
        keys = c.take<unsigned long long>(6);
    });
    if (rc != RT_OK) return rc;
    if (!ctx->update_counts) RT_CUDA(cudaHostAlloc((void**)&ctx->update_counts, 4 * sizeof(int), cudaHostAllocDefault));
    int* flag = rt_bvh_scratch_flag(build);

    const int n3 = 3 * T;
    const unsigned gT = (unsigned)((T + 255) / 256);
    RT_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    const int nc = n3 > u->num_points ? n3 : u->num_points;
    rt_update_check_kernel<<<(unsigned)((nc + 255) / 256), 256, 0, st>>>(u->point_idx, u->points, u->num_points, u->normal_idx,
                                                                         u->normals ? u->num_normals : 0, r->texcoord_idx,
                                                                         r->num_texcoords, r->texture, ctx->scene.meshes + mi,
                                                                         n3, safe_idx, nullptr, safe_tidx, flag);
    RT_CUDA(cudaGetLastError());
    ctx->launches++;
    // the host reads the check before the builder runs: the builder never sees a non-finite key or an unchecked index
    RT_CUDA(cudaMemcpyAsync(ctx->update_counts + 2, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    if (const int bad = ctx->update_counts[2])
    {
        std::string what;
        for (auto b : { std::make_pair(RT_UPD_BAD_POINT_INDEX, "point index"), std::make_pair(RT_UPD_BAD_NORMAL_INDEX, "normal index"),
                        std::make_pair(RT_UPD_BAD_TEXCOORD_INDEX, "texcoord index"), std::make_pair(RT_UPD_BAD_TEXTURE, "texture slot") })
            if (bad & b.first) what += (what.empty() ? " " : ", ") + std::string(b.second);
        std::string msg = std::string(fn) + ":";
        if (!what.empty()) msg += " out of range:" + what;
        if (bad & RT_UPD_BAD_POINT_VALUE) msg += std::string(what.empty() ? "" : ";") + " non-finite point";
        return fail(ctx, RT_ERR_INVALID, msg);
    }
    rc = rt_bvh_build_core(ctx, u->points, safe_idx, T, st, build, ctx->update_counts, ms.spare.nodes, ms.spare.tris, nullptr);
    if (rc != RT_OK) return rc;
    rt_patch_right_child<<<(unsigned)((2 * T - 1 + 255) / 256), 256, 0, st>>>(ms.spare.nodes, 2 * T - 1);
    if (replace)
        rt_replace_shade_kernel<<<gT, 256, 0, st>>>(u->points, safe_idx, u->normals, u->normal_idx, r->texcoords, safe_tidx,
                                                    r->texture, (float*)shade_tmp, T);
    else
        rt_update_shade_kernel<<<gT, 256, 0, st>>>((const float4*)ms.cur.tris, (const float*)ms.cur.shade, u->points, safe_idx,
                                                   u->normals, u->normal_idx, (float*)shade_tmp, T);
    ctx->launches += 2;
    return publish_mesh(ctx, shape, mi, T, u, shade_tmp, keys, nullptr, nullptr, st);
}

// Room for `need` records in a scene array (*ptr: ctx->scene.materials or .lights), enqueued on `st` after the join of
// an update: a larger array from the pool with the first `keep` records copied over.  One an earlier update allocated
// is released with cudaFreeAsync; the uploaded one stays until the next upload or destroy.  Kernels enqueued before the
// update hold the old pointer (DevScene goes to kernels by value) and the join has ordered them before the release.
template <typename T>
static int grow_records(rt_gpu_ctx* ctx, const T** ptr, int* cap, bool* pooled, int need, int keep, cudaStream_t st)
{
    if (need <= *cap) return RT_OK;
    void* p = nullptr;
    int rc = alloc_pooled(ctx, &p, (size_t)need * sizeof(T), st);
    if (rc != RT_OK) return rc;
    if (keep > 0) RT_CUDA(cudaMemcpyAsync(p, *ptr, (size_t)keep * sizeof(T), cudaMemcpyDeviceToDevice, st));
    if (*pooled && (rc = free_pooled(ctx, (void*)*ptr, (size_t)*cap * sizeof(T), st)) != RT_OK) return rc;
    *ptr = (const T*)p; *cap = need; *pooled = true;
    return RT_OK;
}

// count caller records into dst[0, count) on `st`, as kernel parameters
template <typename T>
static int write_records(rt_gpu_ctx* ctx, T* dst, const T* src, int count, cudaStream_t st)
{
    for (int b = 0; b < count; b += RT_RECORDS_PER_LAUNCH)
    {
        const int n = count - b < RT_RECORDS_PER_LAUNCH ? count - b : RT_RECORDS_PER_LAUNCH;
        RecordBatch<T> batch;
        memset(&batch, 0, sizeof batch);
        memcpy(batch.rec, src + b, (size_t)n * sizeof(T));
        rt_update_records_kernel<T><<<1, RT_RECORDS_PER_LAUNCH, 0, st>>>(dst + b, batch, n);
        RT_CUDA(cudaGetLastError());
        ctx->launches++;
    }
    return RT_OK;
}

extern "C" {

int rt_gpu_update_mesh(rt_gpu_ctx* ctx, int32_t shape, const rt_mesh_update* u, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        int mi = -1;
        const int rc = check_mesh_update(ctx, "rt_gpu_update_mesh", shape, u, true, &mi);
        if (rc != RT_OK) return rc;
        const rt_mesh_replace r = { *u, nullptr, 0, nullptr, nullptr };
        return rebuild_mesh(ctx, "rt_gpu_update_mesh", shape, mi, &r, false, stream ? (cudaStream_t)stream : ctx->stream);
    });
}

int rt_gpu_replace_mesh(rt_gpu_ctx* ctx, int32_t shape, const rt_mesh_replace* r, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        const char* fn = "rt_gpu_replace_mesh";
        if (!r) return fail(ctx, ctx->has_scene ? RT_ERR_INVALID : RT_ERR_NO_SCENE, std::string(fn) + ": replace is null");
        int mi = -1;
        int rc = check_mesh_update(ctx, fn, shape, &r->geometry, false, &mi);
        if (rc != RT_OK) return rc;
        if ((r->texcoords == nullptr) != (r->texcoord_idx == nullptr))
            return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": texcoords and texcoord_idx come together");
        if (r->texcoords && r->num_texcoords <= 0) return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": num_texcoords must be positive");
        rc = check_device_args(ctx, fn, { { r->texcoords, "texcoords", 4 }, { r->texcoord_idx, "texcoord_idx", 4 },
                                          { r->texture, "texture", 4 } });
        if (rc != RT_OK) return rc;
        return rebuild_mesh(ctx, fn, shape, mi, r, true, stream ? (cudaStream_t)stream : ctx->stream);
    });
}

// The published topology with new points: O(T) stream-ordered kernels and no host read, so the call returns at once.
// A bad index cannot stop the call on the host; the device publishes a copy of the live set instead (see
// rt_refit_restore_kernel), so the ping-pong stays consistent either way.
int rt_gpu_refit_mesh(rt_gpu_ctx* ctx, int32_t shape, const rt_mesh_update* u, int32_t* status, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        const char* fn = "rt_gpu_refit_mesh";
        int mi = -1;
        int rc = check_mesh_update(ctx, fn, shape, u, true, &mi);
        if (rc != RT_OK) return rc;
        if ((rc = check_device_args(ctx, fn, { { status, "status", 4 } })) != RT_OK) return rc;
        rt_gpu_ctx::MeshState& ms = ctx->mesh_state[mi];
        if (!ms.refittable)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_refit_mesh: the uploaded tree is not a full binary tree whose leaves name every "
                                             "triangle slot once (rt_gpu_update_mesh builds one)");
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        const int T = ms.num_tris, N = 2 * T - 1;
        RT_CUDA(wait_scene(ctx, st));
        if ((rc = alloc_spare(ctx, ms, T, st)) != RT_OK) return rc;
        // scratch: flag, safe point and normal indices (3T each; normals only with normals), shading records in original
        // order (T), bounds keys (6), parent links (N), leaf nodes (T), arrival counters (N)
        int *flag, *safe_p, *safe_n, *parent, *leaf_node, *arrivals; rt_shade* shade_tmp; unsigned long long* keys;
        rc = carve_update_scratch(ctx, st, [&](Carve& c) {
            flag = c.take<int>(1);
            safe_p = c.take<int>(3 * (size_t)T);
            safe_n = u->normals ? c.take<int>(3 * (size_t)T) : nullptr;
            shade_tmp = c.take<rt_shade>((size_t)T);
            keys = c.take<unsigned long long>(6);
            parent = c.take<int>((size_t)N);
            leaf_node = c.take<int>((size_t)T);
            arrivals = c.take<int>((size_t)N);
        });
        if (rc != RT_OK) return rc;
        const unsigned gT = (unsigned)((T + 255) / 256), gN = (unsigned)((N + 255) / 256);

        const int n3 = 3 * T;
        RT_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
        const int nc = n3 > u->num_points ? n3 : u->num_points;
        rt_update_check_kernel<<<(unsigned)((nc + 255) / 256), 256, 0, st>>>(u->point_idx, u->points, u->num_points, u->normal_idx,
                                                                             u->normals ? u->num_normals : 0, nullptr, 0, nullptr,
                                                                             nullptr, n3, safe_p, safe_n, nullptr, flag);
        rt_refit_links_kernel<<<gN, 256, 0, st>>>(ms.cur.nodes, N, parent, leaf_node, arrivals);
        rt_refit_kernel<<<gT, 256, 0, st>>>((const float4*)ms.cur.tris, (const float4*)ms.cur.nodes, u->points, safe_p, leaf_node,
                                            parent, arrivals, ms.spare.tris, (float4*)ms.spare.nodes, T);
        rt_update_shade_kernel<<<gT, 256, 0, st>>>((const float4*)ms.cur.tris, (const float*)ms.cur.shade, u->points, safe_p,
                                                   u->normals, safe_n, (float*)shade_tmp, T);
        RT_CUDA(cudaGetLastError());
        ctx->launches += 4;
        return publish_mesh(ctx, shape, mi, T, u, shade_tmp, keys, flag, status, st);
    });
}

int rt_gpu_update_shapes(rt_gpu_ctx* ctx, const rt_shape* shapes, int32_t first, int32_t count, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_update_shapes before rt_gpu_upload_scene");
        const int num = (int)ctx->host_shapes.size();
        if (first < 0 || count < 0 || first > num || count > num - first)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_shapes: [first, first + count) is not a range of the scene's shapes");
        if (count == 0) return RT_OK;
        if (!shapes) return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_shapes: shapes is null");
        for (int k = 0; k < count; k++)
        {
            const rt_shape& r = shapes[k];
            const rt_shape& up = ctx->host_shapes[first + k];
            if (r.type != up.type || r.mesh != up.mesh || r.has_bounds != up.has_bounds)
                return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_shapes: type, mesh and has_bounds must stay those of the upload");
            if (r.material < -1 || r.material >= (int)ctx->host_materials.size())
                return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_shapes: material index out of range");
        }
        RT_CUDA(cudaSetDevice(ctx->device));
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RT_CUDA(wait_scene(ctx, st));
        int rc = join_scene_readers(ctx, st);
        if (rc != RT_OK) return rc;
        for (int b = 0; b < count; b += RT_SHAPES_PER_LAUNCH)
        {
            const int n = count - b < RT_SHAPES_PER_LAUNCH ? count - b : RT_SHAPES_PER_LAUNCH;
            ShapeBatch batch;
            memset(&batch, 0, sizeof batch);
            memcpy(batch.rec, shapes + b, (size_t)n * sizeof(rt_shape));
            rt_update_shapes_kernel<<<1, RT_SHAPES_PER_LAUNCH, 0, st>>>(const_cast<rt_shape*>(ctx->scene.shapes) + first + b, batch, n);
            RT_CUDA(cudaGetLastError());
            ctx->launches++;
        }
        if ((rc = publish_done(ctx, st)) != RT_OK) return rc;
        for (int k = 0; k < count; k++) ctx->host_shapes[first + k].material = shapes[k].material;
        return RT_OK;
    });
}

int rt_gpu_update_materials(rt_gpu_ctx* ctx, const rt_material* materials, int32_t first, int32_t count, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_update_materials before rt_gpu_upload_scene");
        const int num = (int)ctx->host_materials.size();
        if (first < 0 || count < 0 || first > num || count > 0x7fffffff - first)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_materials: first must be in [0, node count] and count >= 0");
        if (count == 0) return RT_OK;
        if (!materials) return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_materials: materials is null");
        // the checks run on the graph as it will be: an edit can close a cycle through nodes it does not touch
        const int n = std::max(num, first + count);
        std::vector<rt_material> next(ctx->host_materials);
        next.resize((size_t)n);
        std::copy(materials, materials + count, next.begin() + first);
        bool needs_table = false;
        int rc = check_materials(ctx, next.data(), n, "rt_gpu_update_materials: ", &needs_table);
        if (rc != RT_OK) return rc;
        RT_CUDA(cudaSetDevice(ctx->device));
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RT_CUDA(wait_scene(ctx, st));
        if ((rc = join_scene_readers(ctx, st)) != RT_OK) return rc;
        if ((rc = grow_records(ctx, &ctx->scene.materials, &ctx->material_cap, &ctx->materials_pooled, n, num, st)) != RT_OK)
            return rc;
        if ((rc = write_records(ctx, const_cast<rt_material*>(ctx->scene.materials) + first, materials, count, st)) != RT_OK)
            return rc;
        if ((rc = publish_done(ctx, st)) != RT_OK) return rc;
        ctx->host_materials.swap(next);
        ctx->scene.num_materials = n;
        ctx->needs_table = needs_table;
        return RT_OK;
    });
}

int rt_gpu_update_lights(rt_gpu_ctx* ctx, const rt_light* lights, int32_t count, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_update_lights before rt_gpu_upload_scene");
        if (count < 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_lights: count must be >= 0");
        if (count > 0 && !lights) return fail(ctx, RT_ERR_INVALID, "rt_gpu_update_lights: lights is null");
        RT_CUDA(cudaSetDevice(ctx->device));
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RT_CUDA(wait_scene(ctx, st));
        int rc = join_scene_readers(ctx, st);
        if (rc != RT_OK) return rc;
        if ((rc = grow_records(ctx, &ctx->scene.lights, &ctx->light_cap, &ctx->lights_pooled, count, 0, st)) != RT_OK) return rc;
        if ((rc = write_records(ctx, const_cast<rt_light*>(ctx->scene.lights), lights, count, st)) != RT_OK) return rc;
        if ((rc = publish_done(ctx, st)) != RT_OK) return rc;
        ctx->scene.num_lights = count;        // later calls size their Whitted rounds and pools by it
        return RT_OK;
    });
}

int rt_gpu_update_texture(rt_gpu_ctx* ctx, int32_t mesh, int32_t slot, const rt_texture_update* t, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        const std::string f("rt_gpu_update_texture: ");
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_update_texture before rt_gpu_upload_scene");
        if (!t) return fail(ctx, RT_ERR_INVALID, f + "update is null");
        if (mesh < 0 || mesh >= (int)ctx->mesh_textures.size()) return fail(ctx, RT_ERR_INVALID, f + "mesh out of range");
        if (slot < 0 || slot >= (int)ctx->mesh_textures[mesh].size()) return fail(ctx, RT_ERR_INVALID, f + "texture slot out of range");
        const DevTexture dt = ctx->mesh_textures[mesh][slot];
        if (dt.width <= 0 || dt.height <= 0) return fail(ctx, RT_ERR_INVALID, f + "the slot had no pixels at upload");
        if (t->x < 0 || t->y < 0 || t->width < 0 || t->height < 0 || (long long)t->x + t->width > dt.width ||
            (long long)t->y + t->height > dt.height)
            return fail(ctx, RT_ERR_INVALID, f + "rectangle outside the slot");
        if ((t->rgba == nullptr) == (t->texels8 == nullptr)) return fail(ctx, RT_ERR_INVALID, f + "exactly one of rgba and texels8");
        if (t->rgba)
        {
            if (t->pitch < (size_t)t->width * 16 || t->pitch % 4 != 0)
                return fail(ctx, RT_ERR_INVALID, f + "pitch must be at least width * 16 bytes and a multiple of 4");
        }
        else
        {
            if (t->channels != 3 && t->channels != 4) return fail(ctx, RT_ERR_INVALID, f + "texels8 needs 3 or 4 channels");
            if (!t->lut) return fail(ctx, RT_ERR_INVALID, f + "texels8 needs a 512-entry lut");
        }
        RT_CUDA(cudaSetDevice(ctx->device));
        int rc = check_device_args(ctx, "rt_gpu_update_texture", { { t->rgba, "rgba", 4 }, { t->texels8, "texels8", 1 },
                                                                   { t->rgba ? nullptr : t->lut, "lut", 4 } });
        if (rc != RT_OK) return rc;
        if (t->width == 0 || t->height == 0) return RT_OK;
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RT_CUDA(wait_scene(ctx, st));
        if ((rc = join_scene_readers(ctx, st)) != RT_OK) return rc;
        const int ax = dt.x0 + t->x, ay = dt.y0 + t->y;
        if (t->rgba)
            RT_CUDA(cudaMemcpy2DToArrayAsync(ctx->atlas_array, (size_t)ax * 16, (size_t)ay, t->rgba, t->pitch, (size_t)t->width * 16,
                                             (size_t)t->height, cudaMemcpyDeviceToDevice, st));
        else
        {
            const dim3 grid((unsigned)((t->width + 31) / 32), (unsigned)((t->height + 7) / 8));
            rt_expand_texels_kernel<<<grid, dim3(32, 8), 0, st>>>(ctx->atlas_surface, t->texels8, t->lut, t->width, t->height,
                                                                  t->channels, ax, ay);
            RT_CUDA(cudaGetLastError());
            ctx->launches++;
        }
        return publish_done(ctx, st);
    });
}

} // extern "C"
