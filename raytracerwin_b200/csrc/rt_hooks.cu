// rt_hooks.cu — test hooks (arbitrary rays, primitive known-answer tests, texture sampling) and tooling
// (per-round timing) behind include/rt_gpu.h and include/rt_gpu_debug.h.  Not on the render path.
#include "rt_context.hpp"
#include "rt_gpu_debug.h"

// ---- test hooks: arbitrary rays and primitive known-answer tests -------------------------------------------
template <bool CULL>
__global__ void rt_trace_rays_kernel(const DevScene sc, const float* rays, int n, int* shape_out, int* tri_out,
                                     float* hit11, unsigned long long* counters, int exact)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    Ray r; r.o = V3(0, 0, 0); r.d = V3(0, 0, 1); r.dist = 0.0f;
    if (active)
    {
        const float* q = rays + 7 * (size_t)i;
        r.o = V3(q[0], q[1], q[2]); r.d = V3(q[3], q[4], q[5]); r.dist = q[6];
    }
    Hit h; h.pos = V3(0, 0, 0); h.nrm = V3(0, 0, 0); h.dist = 0.0f; h.color = V3(1.0f, 1.0f, 1.0f); h.alpha = 1.0f;
    int tri = -1;
    const int s = trace_scene<CULL>(sc, r, active, false, h, tri, cnt);
    if (active)
    {
        shape_out[i] = s; tri_out[i] = s >= 0 ? tri : -1;
        float* o = hit11 + 11 * (size_t)i;
        for (int k = 0; k < 11; k++) o[k] = 0.0f;
        if (s >= 0)
        {
            o[0] = h.pos.x; o[1] = h.pos.y; o[2] = h.pos.z; o[3] = h.nrm.x; o[4] = h.nrm.y; o[5] = h.nrm.z;
            o[6] = h.dist; o[7] = h.color.x; o[8] = h.color.y; o[9] = h.color.z; o[10] = h.alpha;
        }
    }
    flush_counters(cnt, counters, exact);
}

// kind: 0 aabb (prim 6 floats; out7[0] = tmin), 1 triangle (9), 2 sphere (4), 3 plane (6), 4 capsule (7),
//       5 q_rsqrt (rays unused; prim 1 float; out7[0]), 6 barycentric (prim 12: p,a,b,c; out7[0..2]),
//       7 display (prim 3: linear rgb; flags = ARGB)
__global__ void rt_kat_kernel(int kind, const float* rays, const float* prims, int n, int* flags, float* out7)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Ray r; r.o = V3(0, 0, 0); r.d = V3(0, 0, 1); r.dist = 1.0f;
    if (rays)
    {
        const float* q = rays + 7 * (size_t)i;
        r.o = V3(q[0], q[1], q[2]); r.d = V3(q[3], q[4], q[5]); r.dist = q[6];
    }
    float* o = out7 + 7 * (size_t)i;
    for (int k = 0; k < 7; k++) o[k] = 0.0f;
    float3 pos = V3(0, 0, 0), nrm = V3(0, 0, 0); float dist = 0.0f;
    bool hit = false;
    if (kind == 0)
    {
        const float* b = prims + 6 * (size_t)i;
        RayPre pre = ray_pre(r);
        float tlo, thi;
        hit = slab_general(r, pre, ld3(b), ld3(b + 3), tlo, thi);
        // the walks run slab_fast where this holds; their boxes are finite because the upload refuses other ones
        const bool all_axes = pre.ex && pre.ey && pre.ez && finite3(r.o) && finite3(r.d) && finite3(ld3(b)) && finite3(ld3(b + 3));
        if (all_axes)
        {
            float tlo2, thi2;
            const bool hit2 = slab_fast(r, pre, ld3(b), ld3(b + 3), tlo2, thi2);
            if (hit2 != hit) hit = !hit;   // would surface as a mismatch against the oracle
            // by value: where tlo is a zero (an origin on a face of the box), FMNMX and the reference's ternaries can keep
            // zeros of different sign; no walk can tell them apart (the walks only compare tlo with other values)
            if (hit && tlo2 != tlo) tlo = __uint_as_float(0x7fc00000u);
        }
        flags[i] = hit ? 1 : 0;
        o[0] = hit ? tlo : 0.0f;
        return;
    }
    if (kind == 1)
    {
        const float* t = prims + 9 * (size_t)i;
        const float3 p0 = ld3(t), p1 = ld3(t + 3), p2 = ld3(t + 6);
        const float3 nn = normalized3(cross3(sub3(p1, p0), sub3(p2, p0)));
        hit = triangle_test(r, p0, p1, p2, nn, pos, dist);
        nrm = nn;
    }
    else if (kind == 2) { const float* s = prims + 4 * (size_t)i; hit = sphere_test(r, ld3(s), s[3], pos, nrm, dist); }
    else if (kind == 3) { const float* s = prims + 6 * (size_t)i; hit = plane_test(r, ld3(s), ld3(s + 3), pos, nrm, dist); }
    else if (kind == 4)
    {
        const float* s = prims + 7 * (size_t)i;
        hit = cylinder_test(r, ld3(s), ld3(s + 3), s[6], pos, nrm, dist);
        if (!hit)
        {
            float3 p1, n1, p2, n2; float d1 = 0.0f, d2 = 0.0f;
            const bool b1 = sphere_test(r, ld3(s), s[6], p1, n1, d1);
            const bool b2 = sphere_test(r, ld3(s + 3), s[6], p2, n2, d2);
            hit = b1 || b2;
            if (hit) { const bool first = (b1 && b2) ? (d1 < d2) : b1; pos = first ? p1 : p2; nrm = first ? n1 : n2; dist = first ? d1 : d2; }
        }
    }
    else if (kind == 5) { o[0] = q_rsqrt(prims[i]); flags[i] = 1; return; }
    else if (kind == 6)
    {
        const float* q = prims + 12 * (size_t)i;
        barycentric(ld3(q), ld3(q + 3), ld3(q + 6), ld3(q + 9), o[0], o[1], o[2]);
        flags[i] = 1; return;
    }
    else if (kind == 7) { flags[i] = (int)make_pixel(ld3(prims + 3 * (size_t)i)); return; }
    flags[i] = hit ? 1 : 0;
    if (hit) { o[0] = pos.x; o[1] = pos.y; o[2] = pos.z; o[3] = nrm.x; o[4] = nrm.y; o[5] = nrm.z; o[6] = dist; }
}

__global__ void rt_kat_texture_kernel(cudaTextureObject_t atlas, DevTexture t, const float* uv, int n, float* out4)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 c = texture_sample(atlas, t, uv[2 * i], uv[2 * i + 1]);
    out4[4 * i] = c.x; out4[4 * i + 1] = c.y; out4[4 * i + 2] = c.z; out4[4 * i + 3] = c.w;
}

extern "C" {

/* tooling: entries and walk-kernel time of each round of the last batch / call */
int rt_gpu_debug_rounds(rt_gpu_ctx* ctx, uint32_t* counts, float* ms, int32_t max_rounds)
{
    if (!ctx || !counts || !ms || max_rounds <= 0) return RT_ERR_INVALID;
    RT_CUDA(cudaSetDevice(ctx->device));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    const int n = max_rounds < RT_MAX_ROUNDS ? max_rounds : RT_MAX_ROUNDS;
    RT_CUDA(cudaMemcpy(counts, ctx->pipes[0].round_counters, (size_t)n * sizeof(unsigned), cudaMemcpyDeviceToHost));
    for (int k = 0; k < n; k++)
    {
        ms[k] = 0.0f;
        if (2 * k + 1 < ctx->kev_used) RT_CUDA(cudaEventElapsedTime(&ms[k], ctx->kev[2 * k], ctx->kev[2 * k + 1]));
    }
    unsigned longest = 0;
    RT_CUDA(cudaMemcpy(&longest, ctx->pipes[0].round_counters + RT_MAX_ROUNDS, sizeof(unsigned), cudaMemcpyDeviceToHost));
    if (n > 0) counts[n - 1] = longest;        // last slot: longest single walk (nodes) of the batch
    return ctx->kev_used / 2;
}

/* tooling: begin/end of every timed walk bracket of the last call, in ms since the call began (launch order:
   chunk by chunk, round by round); returns the number of brackets */
int rt_gpu_debug_timeline(rt_gpu_ctx* ctx, float* begin_ms, float* end_ms, int32_t cap)
{
    if (!ctx || !begin_ms || !end_ms || cap <= 0) return RT_ERR_INVALID;
    RT_CUDA(cudaSetDevice(ctx->device));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    const int n = ctx->kev_used / 2 < cap ? ctx->kev_used / 2 : cap;
    for (int k = 0; k < n; k++)
    {
        RT_CUDA(cudaEventElapsedTime(&begin_ms[k], ctx->ev0, ctx->kev[2 * k]));
        RT_CUDA(cudaEventElapsedTime(&end_ms[k], ctx->ev0, ctx->kev[2 * k + 1]));
    }
    return n;
}

/* tooling: long-walk queue sizes per round of the last batch on pipe 0 */
int rt_gpu_debug_long(rt_gpu_ctx* ctx, uint32_t* lcounts, int32_t max_rounds)
{
    if (!ctx || !lcounts || max_rounds <= 0) return RT_ERR_INVALID;
    RT_CUDA(cudaSetDevice(ctx->device));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    const int n = max_rounds < RT_MAX_ROUNDS ? max_rounds : RT_MAX_ROUNDS;
    RT_CUDA(cudaMemcpy(lcounts, ctx->pipes[0].round_counters + 2 * RT_MAX_ROUNDS + 1, (size_t)n * sizeof(unsigned), cudaMemcpyDeviceToHost));
    return RT_OK;
}

int rt_gpu_debug_read_mesh(rt_gpu_ctx* ctx, int32_t mesh, rt_bvh_node* nodes, rt_tri* tris, rt_shade* shade, float* bounds6,
                           float* cull_scale)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_debug_read_mesh before rt_gpu_upload_scene");
        if (mesh < 0 || mesh >= ctx->scene.num_meshes) return fail(ctx, RT_ERR_INVALID, "rt_gpu_debug_read_mesh: mesh out of range");
        RT_CUDA(cudaSetDevice(ctx->device));
        if (ctx->scene_event_live) RT_CUDA(cudaEventSynchronize(ctx->scene_event));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        // the record the kernels read, not the host's bookkeeping
        DevMesh m;
        RT_CUDA(cudaMemcpyAsync(&m, ctx->scene.meshes + mesh, sizeof m, cudaMemcpyDeviceToHost, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        const size_t T = (size_t)m.num_tris;
        if (nodes && m.num_nodes > 0)
            RT_CUDA(cudaMemcpyAsync(nodes, m.nodes, (size_t)m.num_nodes * sizeof(rt_bvh_node), cudaMemcpyDeviceToHost, ctx->stream));
        if (tris && T) RT_CUDA(cudaMemcpyAsync(tris, m.tris, T * sizeof(rt_tri), cudaMemcpyDeviceToHost, ctx->stream));
        if (shade && T) RT_CUDA(cudaMemcpyAsync(shade, m.shade, T * sizeof(rt_shade), cudaMemcpyDeviceToHost, ctx->stream));
        if (bounds6)
        {
            int si = -1;
            for (size_t k = 0; k < ctx->host_shapes.size() && si < 0; k++)
                if (ctx->host_shapes[k].type == RT_SHAPE_MESH && ctx->host_shapes[k].mesh == mesh) si = (int)k;
            if (si < 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_debug_read_mesh: no shape references the mesh");
            rt_shape rec;
            RT_CUDA(cudaMemcpyAsync(&rec, ctx->scene.shapes + si, sizeof rec, cudaMemcpyDeviceToHost, ctx->stream));
            RT_CUDA(cudaStreamSynchronize(ctx->stream));
            for (int c = 0; c < 3; c++) { bounds6[c] = rec.bounds_min[c]; bounds6[3 + c] = rec.bounds_max[c]; }
        }
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        if (cull_scale) *cull_scale = m.cull_scale;
        return RT_OK;
    });
}

int rt_gpu_debug_read_appearance(rt_gpu_ctx* ctx, rt_material* materials, int32_t mat_cap, rt_light* lights, int32_t light_cap,
                                 int32_t* counts2)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_debug_read_appearance before rt_gpu_upload_scene");
        if (mat_cap < 0 || light_cap < 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_debug_read_appearance: negative capacity");
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(wait_scene(ctx, ctx->stream));
        const DevScene& sc = ctx->scene;
        const int nm = std::min(mat_cap, sc.num_materials), nl = std::min(light_cap, sc.num_lights);
        if (materials && nm > 0)
            RT_CUDA(cudaMemcpyAsync(materials, sc.materials, (size_t)nm * sizeof(rt_material), cudaMemcpyDeviceToHost, ctx->stream));
        if (lights && nl > 0)
            RT_CUDA(cudaMemcpyAsync(lights, sc.lights, (size_t)nl * sizeof(rt_light), cudaMemcpyDeviceToHost, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        if (counts2) { counts2[0] = sc.num_materials; counts2[1] = sc.num_lights; }
        return RT_OK;
    });
}

int rt_gpu_debug_read_texture(rt_gpu_ctx* ctx, int32_t mesh, int32_t slot, float* rgba)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_debug_read_texture before rt_gpu_upload_scene");
        if (!rgba || mesh < 0 || mesh >= (int)ctx->mesh_textures.size() || slot < 0 || slot >= (int)ctx->mesh_textures[mesh].size())
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_debug_read_texture: bad arguments");
        const DevTexture t = ctx->mesh_textures[mesh][slot];
        if (t.width <= 0 || t.height <= 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_debug_read_texture: the slot has no pixels");
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(wait_scene(ctx, ctx->stream));
        RT_CUDA(cudaMemcpy2DFromArrayAsync(rgba, (size_t)t.width * 16, ctx->atlas_array, (size_t)t.x0 * 16, (size_t)t.y0,
                                           (size_t)t.width * 16, (size_t)t.height, cudaMemcpyDeviceToHost, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        return RT_OK;
    });
}

int rt_gpu_trace_rays(rt_gpu_ctx* ctx, const float* rays, int32_t n, int32_t traverse, int32_t* shape, int32_t* tri, float* hit11)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_trace_rays before rt_gpu_upload_scene");
        if (n < 0 || (n > 0 && (!rays || !shape || !tri || !hit11))) return fail(ctx, RT_ERR_INVALID, "bad arguments");
        if (n == 0) return RT_OK;
        RT_CUDA(cudaSetDevice(ctx->device));
        float* drays = nullptr; int* dshape = nullptr; int* dtri = nullptr; float* dhit = nullptr;
        RT_CUDA(cudaMalloc((void**)&drays, (size_t)n * 7 * sizeof(float)));
        cudaError_t e = cudaMalloc((void**)&dshape, (size_t)n * sizeof(int));
        if (e == cudaSuccess) e = cudaMalloc((void**)&dtri, (size_t)n * sizeof(int));
        if (e == cudaSuccess) e = cudaMalloc((void**)&dhit, (size_t)n * 11 * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpyAsync(drays, rays, (size_t)n * 7 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = wait_scene(ctx, ctx->stream);
        if (e == cudaSuccess)
        {
            const int exact = traverse == RT_TRAVERSE_EXACT ? 1 : 0;
            if (traverse == RT_TRAVERSE_CULLED)
                rt_trace_rays_kernel<true><<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->scene, drays, n, dshape, dtri, dhit, ctx->counters, exact);
            else
                rt_trace_rays_kernel<false><<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->scene, drays, n, dshape, dtri, dhit, ctx->counters, exact);
            e = cudaGetLastError();
            ctx->launches++;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(shape, dshape, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(tri, dtri, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(hit11, dhit, (size_t)n * 11 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        cudaFree(drays); cudaFree(dshape); cudaFree(dtri); cudaFree(dhit);
        if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, std::string("rt_gpu_trace_rays: ") + cudaGetErrorString(e));
        return RT_OK;
    });
}

int rt_gpu_kat(rt_gpu_ctx* ctx, int32_t kind, const float* rays, const float* prims, int32_t prim_floats, int32_t n,
               int32_t* flags, float* out7)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (n <= 0 || !prims || !flags || !out7 || kind < 0 || kind > 7) return fail(ctx, RT_ERR_INVALID, "bad arguments");
        RT_CUDA(cudaSetDevice(ctx->device));
        float* drays = nullptr; float* dprims = nullptr; int* dflags = nullptr; float* dout = nullptr;
        cudaError_t e = cudaSuccess;
        if (rays) { e = cudaMalloc((void**)&drays, (size_t)n * 7 * sizeof(float)); if (e == cudaSuccess) e = cudaMemcpyAsync(drays, rays, (size_t)n * 7 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream); }
        if (e == cudaSuccess) e = cudaMalloc((void**)&dprims, (size_t)n * prim_floats * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpyAsync(dprims, prims, (size_t)n * prim_floats * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dflags, (size_t)n * sizeof(int));
        if (e == cudaSuccess) e = cudaMalloc((void**)&dout, (size_t)n * 7 * sizeof(float));
        if (e == cudaSuccess)
        {
            rt_kat_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(kind, drays, dprims, n, dflags, dout);
            e = cudaGetLastError();
            ctx->launches++;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(flags, dflags, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out7, dout, (size_t)n * 7 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        cudaFree(drays); cudaFree(dprims); cudaFree(dflags); cudaFree(dout);
        if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, std::string("rt_gpu_kat: ") + cudaGetErrorString(e));
        return RT_OK;
    });
}

int rt_gpu_kat_texture(rt_gpu_ctx* ctx, int32_t texture, const float* uv, int32_t n, float* out4)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "no scene");
        if (texture < 0 || texture >= (int)ctx->host_textures.size() || n <= 0 || !uv || !out4) return fail(ctx, RT_ERR_INVALID, "bad arguments");
        RT_CUDA(cudaSetDevice(ctx->device));
        float* duv = nullptr; float* dout = nullptr;
        cudaError_t e = cudaMalloc((void**)&duv, (size_t)n * 2 * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc((void**)&dout, (size_t)n * 4 * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpyAsync(duv, uv, (size_t)n * 2 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = wait_scene(ctx, ctx->stream);      // after every rt_gpu_update_texture enqueued so far
        if (e == cudaSuccess)
        {
            rt_kat_texture_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->scene.atlas, ctx->host_textures[texture], duv, n, dout);
            e = cudaGetLastError();
            ctx->launches++;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(out4, dout, (size_t)n * 4 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        cudaFree(duv); cudaFree(dout);
        if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, std::string("rt_gpu_kat_texture: ") + cudaGetErrorString(e));
        return RT_OK;
    });
}

} // extern "C"
