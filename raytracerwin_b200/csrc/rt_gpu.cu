// rt_gpu.cu — the B200 (sm_100a) implementation behind include/rt_gpu.h.
//
// Replaces ThreadWorker_Render + everything beneath it (RayTracerProgram.cpp:131-188,
// RayTracerScene.cpp:31-175, KdTree.cpp:128-232, MeshShape.cpp:280-331, SurfaceMaterials.cpp,
// RRay.cpp, Texture.cpp:23-57) and the ThreadTaskQueue dispatch (ThreadTaskQueue.h) that feeds it.
//
// Execution model (not the reference's): a WAVEFRONT.  The work list of a render call is every
// (sample, pixel) pair, enumerated as 8x4-pixel blocks so that a warp gets coherent camera rays.
//   generate  one thread per item: camera ray, shape list up to the first mesh whose bounds the ray
//             enters.  Rays that end there having hit nothing (most: they see the sky) are retired
//             on the spot at full warp width; the rest become PATHS — a record in a pool, an entry
//             in the round-0 queue, compacted per warp with __ballot_sync/__popc/__shfl_sync.
//   walk      persistent warps pop path ids from the round's queue and walk the mesh (the
//             reference's KdNode recursion, flattened); a lane that finishes pops the next id, so
//             live walks stay packed in full warps although one ray visits 3 nodes and its
//             neighbour 2000.  Round 0 (camera rays, coherent) is walked by the packet kernel
//             instead — a warp's 32 rays share one node fetch per step — and walks that would hold
//             a round (very long ones, thin rounds) by the long-walk kernel, a warp per walk.
//   shade     one thread per queue entry: hit attributes, texture, rest of the shape list, material
//             bounce / alpha / light loop; ends the path (fold + sample) or starts its next segment
//             and pushes it — ballot-compacted again — into the next round's queue.
// walk and shade alternate once per (segment x mesh); nothing returns to the host in between.
// Each finished path writes one float4 radiance sample; a streaming kernel folds the samples of a
// pixel into accuBuffer[] in the reference's order (4 sub-samples -> /4 -> AddPixel per pass,
// RayTracerProgram.cpp:155-185), which keeps the accumulation bit-identical for any GPU count and
// any scheduling.
//
// The whole file is compiled with -fmad=false; see rt_device.cuh.
#include "rt_context.hpp"
#include "rt_wave_kernels.cuh"

thread_local std::string g_create_error;

// for rt_bvh_build.cu, which does not see the context's layout (library-internal: not exported)
__attribute__((visibility("hidden"))) int rt_ctx_device(rt_gpu_ctx* ctx) { return ctx ? ctx->device : -1; }
__attribute__((visibility("hidden"))) void rt_ctx_set_error(rt_gpu_ctx* ctx, const char* msg) { if (ctx && msg) ctx->err = msg; }

// The binary tree collapsed into nodes of up to eight children for rt_walk_octo_kernel: out holds 8 records per
// node, {bmin, ref}{bmax, count} (count in record 0), children in pre-order = slot order; ref >= 0: child node,
// ref < 0: ~leaf slot.  A node starts with its two children and keeps replacing the inner child with the largest
// subtree by that child's two children until it has eight (or only leaves).
static void build_octo(const rt_bvh_node* nodes, int n, std::vector<rt_bvh_node>& out)
{
    out.clear();
    if (n <= 0) return;
    struct Job { int binary; int slot; };           // wide node `slot` collapses the subtree of binary node `binary`
    std::vector<Job> jobs;
    auto new_node = [&]() { const int k = (int)(out.size() / 8); out.resize(out.size() + 8); return k; };
    jobs.push_back(Job{ 0, new_node() });
    while (!jobs.empty())
    {
        const Job j = jobs.back(); jobs.pop_back();
        int kids[8], nk = 0;
        if (nodes[j.binary].tri >= 0) kids[nk++] = j.binary;                 // a tree of one leaf
        else { kids[nk++] = j.binary + 1; kids[nk++] = nodes[j.binary + 1].escape; }
        for (;;)
        {
            int pick = -1, size = 1;
            for (int c = 0; c < nk; c++)
                if (nodes[kids[c]].tri < 0 && nodes[kids[c]].escape - kids[c] > size) { pick = c; size = nodes[kids[c]].escape - kids[c]; }
            if (pick < 0 || nk == 8) break;
            const int b = kids[pick];
            for (int c = nk; c > pick + 1; c--) kids[c] = kids[c - 1];
            kids[pick] = b + 1; kids[pick + 1] = nodes[b + 1].escape;
            nk++;
        }
        for (int c = 0; c < 8; c++)
        {
            rt_bvh_node rec;
            memset(&rec, 0, sizeof rec);
            rec.escape = ~0;                                        // (unused slot: a leaf ref that is never looked at)
            if (c < nk)
            {
                const rt_bvh_node& b = nodes[kids[c]];
                for (int x = 0; x < 3; x++) { rec.bmin[x] = b.bmin[x]; rec.bmax[x] = b.bmax[x]; }
                if (b.tri >= 0) rec.escape = ~b.tri;
                else { const int child = new_node(); rec.escape = child; jobs.push_back(Job{ kids[c], child }); }
            }
            rec.tri = nk;                                           // every record carries the count; record 0's is read
            out[(size_t)j.slot * 8 + c] = rec;
        }
    }
}

static inline bool texture_has_pixels(const rt_texture& t) { return t.rgba != nullptr || t.texels8 != nullptr; }

// RTexture::LoadTexturePNG's texel loop (Texture.cpp:119-151) on the device: 8-bit code -> table entry.  The
// table is the host's (glibc powf(c / 255, 2.2f) for rgb, c / 255 for alpha), so the float4 texels written into
// the atlas are the reference's bit for bit.
__global__ void rt_expand_texels_kernel(cudaSurfaceObject_t atlas, const uint8_t* __restrict__ texels, const float* __restrict__ lut,
                                        int width, int height, int channels, int x0, int y0)
{
    __shared__ float s_lut[512];
    for (int i = threadIdx.y * 32 + threadIdx.x; i < 512; i += 256) s_lut[i] = lut[i];
    __syncthreads();
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= width || y >= height) return;
    const uint8_t* p = texels + ((size_t)y * width + x) * channels;
    const float4 v = make_float4(s_lut[p[0]], s_lut[p[1]], s_lut[p[2]], channels == 4 ? s_lut[256 + p[3]] : 1.0f);
    surf2Dwrite(v, atlas, (x0 + x) * 16, y0 + y);
}

__global__ void rt_shade_leaf_order_kernel(const float4* __restrict__ tris, const float4* __restrict__ shade, float4* __restrict__ out, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int index = __float_as_int(tris[4 * (size_t)k].w);        // rt_tri.index: the triangle's place in the original order
#pragma unroll
    for (int j = 0; j < 4; j++) out[4 * (size_t)k + j] = shade[4 * (size_t)index + j];
}

static void free_scene(rt_gpu_ctx* ctx)
{
    for (cudaTextureObject_t t : ctx->texobjs) cudaDestroyTextureObject(t);
    for (cudaArray_t a : ctx->arrays) cudaFreeArray(a);
    for (void* p : ctx->scene_allocs) cudaFree(p);
    ctx->texobjs.clear(); ctx->arrays.clear(); ctx->scene_allocs.clear(); ctx->host_textures.clear();
    ctx->has_scene = false; ctx->scene_bytes = 0;
    memset(&ctx->scene, 0, sizeof ctx->scene);
}

// the context stream and every pipe: nothing of this context is running afterwards
static cudaError_t sync_all_streams(rt_gpu_ctx* ctx)
{
    cudaError_t first = ctx->stream ? cudaStreamSynchronize(ctx->stream) : cudaSuccess;
    for (int k = 0; k < RT_PIPES; k++)
        if (ctx->pipes[k].stream)
        {
            const cudaError_t e = cudaStreamSynchronize(ctx->pipes[k].stream);
            if (first == cudaSuccess) first = e;
        }
    for (int k = 0; k < RT_FRAME_SLOTS; k++)
        if (k != ctx->slot && ctx->parked[k].stream)
        {
            const cudaError_t e = cudaStreamSynchronize(ctx->parked[k].stream);
            if (first == cudaSuccess) first = e;
        }
    return first;
}

// frame slots: the live members of the context <-> a parked set
static void park_slot(rt_gpu_ctx* ctx, rt_gpu_ctx::FrameSlot& f)
{
    f.stream = ctx->stream; f.ev0 = ctx->ev0; f.ev1 = ctx->ev1; f.timed = ctx->timed;
    f.width = ctx->width; f.height = ctx->height;
    f.accum = ctx->accum; f.display = ctx->display; f.prim_ids = ctx->prim_ids; f.prim_dist = ctx->prim_dist; f.preview = ctx->preview;
}

static void unpark_slot(rt_gpu_ctx* ctx, const rt_gpu_ctx::FrameSlot& f)
{
    ctx->stream = f.stream; ctx->ev0 = f.ev0; ctx->ev1 = f.ev1; ctx->timed = f.timed;
    ctx->width = f.width; ctx->height = f.height;
    ctx->accum = f.accum; ctx->display = f.display; ctx->prim_ids = f.prim_ids; ctx->prim_dist = f.prim_dist; ctx->preview = f.preview;
}

static void free_frame(rt_gpu_ctx* ctx)
{
    cudaFree(ctx->accum); cudaFree(ctx->display); cudaFree(ctx->prim_ids); cudaFree(ctx->prim_dist); cudaFree(ctx->preview);
    ctx->accum = nullptr; ctx->display = nullptr; ctx->prim_ids = nullptr; ctx->prim_dist = nullptr; ctx->preview = nullptr;
    ctx->width = ctx->height = 0;
}

template <typename T>
static int upload(rt_gpu_ctx* ctx, const T* src, size_t count, T** out)
{
    *out = nullptr;
    if (count == 0) return RT_OK;
    void* p = nullptr;
    RT_CUDA(cudaMalloc(&p, count * sizeof(T)));
    ctx->scene_allocs.push_back(p);
    ctx->scene_bytes += count * sizeof(T);
    RT_CUDA(cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    *out = (T*)p;
    return RT_OK;
}

template <bool CULL>
static cudaError_t launch_generate(int mode, unsigned grid, cudaStream_t st, const DevScene& sc, const RenderArgs& a, const WaveArgs& w)
{
    switch (mode)
    {
    case RT_MODE_PATH: rt_generate_kernel<CULL, RT_MODE_PATH><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_MODE_PREVIEW: rt_generate_kernel<CULL, RT_MODE_PREVIEW><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_MODE_WHITTED: rt_generate_kernel<CULL, RT_MODE_WHITTED><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_MODE_PRIMARY: rt_generate_kernel<CULL, RT_MODE_PRIMARY><<<grid, 256, 0, st>>>(sc, a, w); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

template <bool CULL>
static cudaError_t launch_shade(int mode, unsigned grid, cudaStream_t st, const DevScene& sc, const RenderArgs& a, const WaveArgs& w, int round)
{
    switch (mode)
    {
    case RT_MODE_PATH: rt_shade_kernel<CULL, RT_MODE_PATH><<<grid, 256, 0, st>>>(sc, a, w, round); break;
    case RT_MODE_PREVIEW: rt_shade_kernel<CULL, RT_MODE_PREVIEW><<<grid, 256, 0, st>>>(sc, a, w, round); break;
    case RT_MODE_WHITTED: rt_shade_kernel<CULL, RT_MODE_WHITTED><<<grid, 256, 0, st>>>(sc, a, w, round); break;
    case RT_MODE_PRIMARY: rt_shade_kernel<CULL, RT_MODE_PRIMARY><<<grid, 256, 0, st>>>(sc, a, w, round); break;
    case RT_QMODE_NEAREST: rt_shade_kernel<CULL, RT_QMODE_NEAREST><<<grid, 256, 0, st>>>(sc, a, w, round); break;
    case RT_QMODE_ANY: rt_shade_kernel<CULL, RT_QMODE_ANY><<<grid, 256, 0, st>>>(sc, a, w, round); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

template <bool CULL>
static cudaError_t launch_query_generate(int mode, unsigned grid, cudaStream_t st, const DevScene& sc, const RenderArgs& a, const WaveArgs& w)
{
    switch (mode)
    {
    case RT_QMODE_NEAREST: rt_query_generate_kernel<CULL, RT_QMODE_NEAREST><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_QMODE_ANY: rt_query_generate_kernel<CULL, RT_QMODE_ANY><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_MODE_PATH: rt_query_generate_kernel<CULL, RT_MODE_PATH><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_MODE_PREVIEW: rt_query_generate_kernel<CULL, RT_MODE_PREVIEW><<<grid, 256, 0, st>>>(sc, a, w); break;
    case RT_MODE_WHITTED: rt_query_generate_kernel<CULL, RT_MODE_WHITTED><<<grid, 256, 0, st>>>(sc, a, w); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

template <bool CULL>
static cudaError_t launch_finish(int mode, unsigned grid, cudaStream_t st, const DevScene& sc, const RenderArgs& a, const WaveArgs& w, int round)
{
    switch (mode)
    {
    case RT_MODE_PATH: rt_finish_kernel<CULL, RT_MODE_PATH><<<grid, 128, 0, st>>>(sc, a, w, round); break;
    case RT_MODE_PREVIEW: rt_finish_kernel<CULL, RT_MODE_PREVIEW><<<grid, 128, 0, st>>>(sc, a, w, round); break;
    case RT_MODE_WHITTED: rt_finish_kernel<CULL, RT_MODE_WHITTED><<<grid, 128, 0, st>>>(sc, a, w, round); break;
    case RT_MODE_PRIMARY: rt_finish_kernel<CULL, RT_MODE_PRIMARY><<<grid, 128, 0, st>>>(sc, a, w, round); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

static cudaError_t launch_walk(bool cull, bool top, unsigned grid, cudaStream_t st, const DevScene& sc, const RenderArgs& a, const WaveArgs& w, int round, int resumed)
{
    if (cull) { if (top) rt_walk_kernel<true, true><<<grid, 256, 0, st>>>(sc, a, w, round, resumed); else rt_walk_kernel<true, false><<<grid, 256, 0, st>>>(sc, a, w, round, resumed); }
    else { if (top) rt_walk_kernel<false, true><<<grid, 256, 0, st>>>(sc, a, w, round, resumed); else rt_walk_kernel<false, false><<<grid, 256, 0, st>>>(sc, a, w, round, resumed); }
    return cudaGetLastError();
}

template <typename T>
static cudaError_t grow(T** ptr, size_t* cap, size_t need)
{
    if (need <= *cap) return cudaSuccess;
    cudaFree(*ptr); *ptr = nullptr; *cap = 0;
    cudaError_t e = cudaMalloc((void**)ptr, need * sizeof(T));
    if (e == cudaSuccess) *cap = need;
    return e;
}

// resident CTAs per SM of the walk kernels (persistent grids), queried once
static int init_walk_grid(rt_gpu_ctx* ctx)
{
    if (ctx->walk_blocks_per_sm != 0) return RT_OK;
    int b0 = 0, b1 = 0;
    RT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b0, rt_walk_kernel<true, true>, 256, 0));
    RT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b1, rt_walk_kernel<false, true>, 256, 0));
    ctx->walk_blocks_per_sm = b0 < b1 ? b0 : b1;
    RT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->octo_blocks_per_sm, rt_walk_octo_kernel, 256, 0));
    if (ctx->octo_blocks_per_sm < 1) return fail(ctx, RT_ERR_CUDA, "8-wide walk kernel does not fit on an SM");
    if (ctx->walk_blocks_per_sm < 1) return fail(ctx, RT_ERR_CUDA, "walk kernel does not fit on an SM");
    return RT_OK;
}

// Path pools (one per pipe; render_tile and rt_gpu_query_rays share them).  plan_pools: the records a batch of
// `batch` items may use — all of them up to the per-pipe maximum, fewer when the pools have to grow and half of
// the free device memory cannot hold that many (a smaller pool only costs retry passes or smaller query chunks).
// grow_pools then makes the pools at least that large, with `levels` unwinding levels and the Whitted fields if
// asked; it only ever grows them, and synchronises only when it does.
static int plan_pools(rt_gpu_ctx* ctx, size_t batch, size_t levels, bool whitted, size_t* out_want)
{
    size_t pool_want = batch < ctx->max_pool_paths ? batch : ctx->max_pool_paths;
    if (pool_want > ctx->pool_cap || levels > ctx->pool_levels || (whitted && !ctx->pool_whitted))
    {
        // (only when the pools have to grow: the memory query costs a driver round trip)
        // keep all pools together within ~half of the device memory that is free right now (deep bounce
        // budgets make a path record large: 36 B per level); a smaller pool only costs retry passes
        const size_t lv = levels > ctx->pool_levels ? levels : ctx->pool_levels;
        const size_t per_path = 9 * 16 + ((whitted || ctx->pool_whitted) ? 64 : 0) + lv * 36 + 12;
        size_t free_b = 0, total_b = 0;
        RT_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t have_b = free_b + ctx->pool_cap * (9 * 16 + (ctx->pool_whitted ? 64 : 0) + ctx->pool_levels * 36 + 12) * RT_PIPES;
        const size_t fit = have_b / 2 / RT_PIPES / per_path;
        if (pool_want > fit) pool_want = fit > 255 ? (fit & ~(size_t)255) : fit;
        if (pool_want < (batch < 4096 ? batch : (size_t)4096)) return fail(ctx, RT_ERR_NOMEM, "not enough device memory for the path pools");
    }
    *out_want = pool_want;
    return RT_OK;
}

static int grow_pools(rt_gpu_ctx* ctx, size_t pool_want, size_t levels, bool whitted)
{
    if (!(pool_want > ctx->pool_cap || levels > ctx->pool_levels || (whitted && !ctx->pool_whitted))) return RT_OK;
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    const bool same_shape = levels <= ctx->pool_levels && (!whitted || ctx->pool_whitted);
    const size_t cap = (same_shape && ctx->pool_cap > pool_want) ? ctx->pool_cap : pool_want;
    const size_t lv = levels > ctx->pool_levels ? levels : ctx->pool_levels;
    const bool wh = whitted || ctx->pool_whitted;
    for (int k = 0; k < RT_PIPES; k++)
    {
        rt_gpu_ctx::Pipe& pp = ctx->pipes[k];
        RT_CUDA(cudaStreamSynchronize(pp.stream));
        for (void* q : pp.allocs) cudaFree(q);
        pp.allocs.clear();
        auto alloc = [&](size_t bytes, void** out) -> cudaError_t {
            cudaError_t e = cudaMalloc(out, bytes);
            if (e == cudaSuccess) pp.allocs.push_back(*out);
            return e;
        };
        PathPool& pl = pp.pool;
        memset(&pl, 0, sizeof pl);
        RT_CUDA(alloc(cap * 16, (void**)&pl.ro)); RT_CUDA(alloc(cap * 16, (void**)&pl.rd));
        RT_CUDA(alloc(cap * 16, (void**)&pl.cur)); RT_CUDA(alloc(cap * 16, (void**)&pl.bp));
        RT_CUDA(alloc(cap * 16, (void**)&pl.h0)); RT_CUDA(alloc(cap * 16, (void**)&pl.h1));
        RT_CUDA(alloc(cap * 16, (void**)&pl.h2)); RT_CUDA(alloc(cap * 16, (void**)&pl.pa));
        RT_CUDA(alloc(cap * 16, (void**)&pl.pb));
        if (wh)
        {
            RT_CUDA(alloc(cap * 16, (void**)&pl.w0)); RT_CUDA(alloc(cap * 16, (void**)&pl.w1));
            RT_CUDA(alloc(cap * 16, (void**)&pl.w2)); RT_CUDA(alloc(cap * 16, (void**)&pl.w3));
        }
        RT_CUDA(alloc(cap * lv * 16, (void**)&pl.st0)); RT_CUDA(alloc(cap * lv * 16, (void**)&pl.st1));
        RT_CUDA(alloc(cap * lv * 4, (void**)&pl.st2));
        RT_CUDA(alloc(cap * 4, (void**)&pp.queue[0])); RT_CUDA(alloc(cap * 4, (void**)&pp.queue[1]));
        RT_CUDA(alloc(cap * 4, (void**)&pp.longq));
        RT_CUDA(alloc(cap * 4, (void**)&pp.slowq));
        pl.cap = (unsigned)cap;
    }
    ctx->pool_cap = cap; ctx->pool_levels = lv; ctx->pool_whitted = wh;
    return RT_OK;
}

// the wavefront arguments of one pipe: its pool, queues and round counters, and the scheduling knobs
static WaveArgs pipe_wave_args(const rt_gpu_ctx* ctx, const rt_gpu_ctx::Pipe& pp, int packets)
{
    WaveArgs w;
    memset(&w, 0, sizeof w);
    w.pool = pp.pool;
    w.queue[0] = pp.queue[0]; w.queue[1] = pp.queue[1];
    w.counts = pp.round_counters; w.heads = pp.round_counters + RT_MAX_ROUNDS + 1;
    w.longq = pp.longq; w.lcounts = w.heads + RT_MAX_ROUNDS; w.lheads = w.lcounts + RT_MAX_ROUNDS;
    w.slowq = pp.slowq; w.scounts = w.lheads + RT_MAX_ROUNDS; w.sheads = w.scounts + RT_MAX_ROUNDS;
    w.packet_probe = ctx->tune_packet_probe; w.packet_min_lanes = ctx->tune_packet_min_lanes;
    w.long_limit = ctx->tune_long_limit; w.small_round = ctx->tune_small_round;
    w.thin_count = ctx->tune_thin_count; w.thin_limit = ctx->tune_thin_limit;
    w.packets = packets;
    w.min_lanes = ctx->tune_min_lanes; w.leaf_wait = ctx->tune_leaf_wait; w.window = ctx->tune_window;
    return w;
}

// Work forked from a caller's stream onto the pipes: any error return before the join leaves pipes with work in
// flight that the caller's stream has not been ordered after; wait for them on the way out, so that a later reset /
// readback / upload cannot race them.
struct PipeGuard
{
    rt_gpu_ctx* ctx;
    bool used[RT_PIPES];
    bool joined;
    ~PipeGuard()
    {
        if (joined) return;
        for (int k = 0; k < RT_PIPES; k++)
            if (used[k]) cudaStreamSynchronize(ctx->pipes[k].stream);
    }
};

// One round of the wavefront on a pipe: the mesh walks of the round's queue (rounds below `packet_rounds` as packets,
// then the walks they hand back lane by lane; later rounds lane by lane or on the 8-wide tree), the long walks parked
// on the way, then the shade kernel in `mode`.  small_pass / thin: the reduced grids of render_tile's retry passes
// and of late rounds with frames in flight.  mark(class, stream) tags each launch for rt_gpu_time_kernels(ctx, 2);
// `timed` lets the walk brackets of rt_gpu_time_kernels(ctx, 1) be recorded.
template <typename Mark>
static int enqueue_round(rt_gpu_ctx* ctx, rt_gpu_ctx::Pipe& pp, const RenderArgs& a, const WaveArgs& w, int mode, int round,
                         bool cull, int packet_rounds, bool has_mesh, bool small_pass, bool thin, unsigned walk_grid,
                         unsigned shade_grid, bool timed, Mark& mark)
{
    const unsigned sms = (unsigned)ctx->num_sms;
    if (has_mesh)
    {
        if (timed && ctx->time_walks)
        {
            while ((int)ctx->kev.size() < ctx->kev_used + 2)
            {
                cudaEvent_t e = nullptr;
                RT_CUDA(cudaEventCreate(&e));
                ctx->kev.push_back(e);
            }
            RT_CUDA(cudaEventRecord(ctx->kev[ctx->kev_used], pp.stream));
        }
        if (round < packet_rounds)
        {
            // packets first; what they hand back (incoherent ones) goes on lane by lane
            RT_CUDA(mark(RT_KERNEL_PACKET_WALK, pp.stream));
            if (cull) rt_walk_packet_kernel<true><<<small_pass ? sms : walk_grid, 256, 0, pp.stream>>>(ctx->scene, a, w, round);
            else rt_walk_packet_kernel<false><<<small_pass ? sms : walk_grid, 256, 0, pp.stream>>>(ctx->scene, a, w, round);
            RT_CUDA(cudaGetLastError());
            ctx->launches++;
            RT_CUDA(mark(RT_KERNEL_WALK, pp.stream));
            RT_CUDA(launch_walk(cull, ctx->tune_top_stage, small_pass ? sms : walk_grid, pp.stream, ctx->scene, a, w, round, 1));
        }
        else if (cull && ctx->tune_octo)
        {
            // bounce / shadow rounds of the culled traversal: the 8-wide tree
            RT_CUDA(mark(RT_KERNEL_WALK, pp.stream));
            rt_walk_octo_kernel<<<(unsigned)(ctx->num_sms * ctx->octo_blocks_per_sm), 256, 0, pp.stream>>>(ctx->scene, a, w, round);
        }
        else
        {
            RT_CUDA(mark(RT_KERNEL_WALK, pp.stream));
            RT_CUDA(launch_walk(cull, ctx->tune_top_stage, small_pass ? sms : (thin ? walk_grid / 4u : walk_grid), pp.stream, ctx->scene, a, w, round, 0));
        }
        RT_CUDA(cudaGetLastError());
        const bool time_long = ctx->tune_time_long;     // tooling: bracket walk + long walk
        if (timed && ctx->time_walks && !time_long)
        {
            RT_CUDA(cudaEventRecord(ctx->kev[ctx->kev_used + 1], pp.stream));
            ctx->kev_used += 2;
        }
        ctx->launches++;
        // the walks that kernel parked as too long, one warp each
        RT_CUDA(mark(RT_KERNEL_LONG_WALK, pp.stream));
        {
            const int group = ctx->tune_long_group;
            const unsigned lgrid = (unsigned)ctx->num_sms * ((thin || small_pass) ? 1u : (unsigned)RT_LONG_BLOCKS);
#define RT_LAUNCH_LONG(G) (cull ? rt_longwalk_kernel<true, G><<<lgrid, 256, 0, pp.stream>>>(ctx->scene, a, w, round) \
                                : rt_longwalk_kernel<false, G><<<lgrid, 256, 0, pp.stream>>>(ctx->scene, a, w, round))
            if (group == 32) RT_LAUNCH_LONG(32); else if (group == 16) RT_LAUNCH_LONG(16); else RT_LAUNCH_LONG(8);
#undef RT_LAUNCH_LONG
        }
        RT_CUDA(cudaGetLastError());
        if (timed && ctx->time_walks && time_long)
        {
            RT_CUDA(cudaEventRecord(ctx->kev[ctx->kev_used + 1], pp.stream));
            ctx->kev_used += 2;
        }
        ctx->launches++;
    }
    RT_CUDA(mark(RT_KERNEL_SHADE, pp.stream));
    const unsigned sgrid = small_pass ? (sms < shade_grid ? sms : shade_grid) : (thin ? (shade_grid + 7u) / 8u : shade_grid);
    RT_CUDA(cull ? launch_shade<true>(mode, sgrid, pp.stream, ctx->scene, a, w, round)
                 : launch_shade<false>(mode, sgrid, pp.stream, ctx->scene, a, w, round));
    ctx->launches++;
    return RT_OK;
}

// rt_gpu_query_rays / rt_gpu_radiance_rays take device memory of the context's GPU only
static bool on_device(const rt_gpu_ctx* ctx, const void* ptr)
{
    cudaPointerAttributes at;
    memset(&at, 0, sizeof at);
    const cudaError_t e = cudaPointerGetAttributes(&at, ptr);
    if (e != cudaSuccess) cudaGetLastError();
    return e == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && at.device == ctx->device;
}

// A batch of n caller rays through the render's wavefront, ordered on `st`: query generate in `mode`, then `rounds`
// rounds (walks + long walks + shade in `mode`) on the pipes' pools and queues.  The batch is cut into pieces of
// `piece` rays (a multiple of 32 that fits a pool, so that round-0 packets stay 32 consecutive rays of the caller's
// order) and the pieces are dealt round-robin to the pipes, so that the tail of one overlaps the next.
// set_piece(a, begin, count) points the argument block at the piece's part of the caller's arrays.  Nothing that a
// later render reads is touched: frame buffers and slot, ev0 / ev1, the pipe cursor and the round sizes remembered
// per pipe (the quarter grids they steer are for frames in flight; a query round gets the full grids).
template <typename SetPiece>
static int enqueue_ray_batch(rt_gpu_ctx* ctx, RenderArgs& a, size_t n, size_t piece, int mode, int rounds, bool has_mesh,
                             bool cull, cudaStream_t st, SetPiece set_piece)
{
    const int packet_rounds = ctx->tune_packet_rounds >= 0 ? ctx->tune_packet_rounds : 1;
    const unsigned walk_grid = (unsigned)(ctx->num_sms * ctx->walk_blocks_per_sm);
    const int npipes = ctx->tune_pipes;
    auto no_mark = [](int, cudaStream_t) -> cudaError_t { return cudaSuccess; };
    RT_CUDA(cudaEventRecord(ctx->fork, st));
    PipeGuard guard = { ctx, { false }, false };
    int index = 0;
    for (size_t begin = 0; begin < n; begin += piece, index++)
    {
        const size_t count = n - begin < piece ? n - begin : piece;
        const int pipe = index % npipes;
        rt_gpu_ctx::Pipe& pp = ctx->pipes[pipe];
        if (!guard.used[pipe]) { RT_CUDA(cudaStreamWaitEvent(pp.stream, ctx->fork, 0)); guard.used[pipe] = true; }
        a.q_count = (int)count;
        set_piece(a, begin, count);
        WaveArgs w = pipe_wave_args(ctx, pp, packet_rounds > 0 && has_mesh ? 1 : 0);
        w.item_count = (unsigned)count;
        unsigned gen_grid = (unsigned)((count + 255) / 256);
        if (gen_grid > (unsigned)ctx->num_sms * 8u) gen_grid = (unsigned)ctx->num_sms * 8u;
        unsigned shade_grid = (unsigned)((count + 255) / 256);
        if (shade_grid > (unsigned)ctx->num_sms * 16u) shade_grid = (unsigned)ctx->num_sms * 16u;
        RT_CUDA(cudaMemsetAsync(pp.round_counters, 0, (6 * RT_MAX_ROUNDS + 1) * sizeof(unsigned), pp.stream));
        RT_CUDA(cull ? launch_query_generate<true>(mode, gen_grid, pp.stream, ctx->scene, a, w)
                     : launch_query_generate<false>(mode, gen_grid, pp.stream, ctx->scene, a, w));
        ctx->launches++;
        for (int round = 0; round < rounds; round++)
        {
            const int rc = enqueue_round(ctx, pp, a, w, mode, round, cull, packet_rounds, has_mesh, false, false,
                                         walk_grid, shade_grid, false, no_mark);
            if (rc != RT_OK) return rc;
        }
        RT_CUDA(cudaEventRecord(pp.done, pp.stream));
    }
    // join: `st` continues after every pipe
    for (int k = 0; k < RT_PIPES; k++)
        if (guard.used[k]) RT_CUDA(cudaStreamWaitEvent(st, ctx->pipes[k].done, 0));
    guard.joined = true;
    return RT_OK;
}

extern "C" {

int rt_gpu_abi_version(void) { return RT_GPU_ABI_VERSION; }

int rt_gpu_device_count(void)
{
    return rt_guard(nullptr, [&]() -> int {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
        return n;
    });
}

static void tuning_from_env(rt_gpu_ctx* ctx);
int rt_gpu_create(int device, rt_gpu_ctx** out_ctx)
{
    rt_gpu_ctx* ctx = nullptr;
    if (!out_ctx) return fail(nullptr, RT_ERR_INVALID, "out_ctx is null");
    *out_ctx = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, RT_ERR_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") +
                                              (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= n) return fail(nullptr, RT_ERR_INVALID, "device index out of range");
    RT_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RT_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, RT_ERR_CUDA, "device is not sm_100 (this library carries sm_100a code only)");
    ctx = new rt_gpu_ctx();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    memset(&ctx->scene, 0, sizeof ctx->scene);
    cudaError_t e2 = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaEventCreate(&ctx->ev0);
    if (e2 == cudaSuccess) e2 = cudaEventCreate(&ctx->ev1);
    if (e2 == cudaSuccess) e2 = cudaMalloc((void**)&ctx->counters, sizeof(rt_counters));
    if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&ctx->fork, cudaEventDisableTiming);
    for (int k = 0; k < RT_PIPES && e2 == cudaSuccess; k++)
    {
        e2 = cudaStreamCreateWithFlags(&ctx->pipes[k].stream, cudaStreamNonBlocking);
        if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&ctx->pipes[k].done, cudaEventDisableTiming);
        if (e2 == cudaSuccess) e2 = cudaMalloc((void**)&ctx->pipes[k].round_counters, (6 * RT_MAX_ROUNDS + 1) * sizeof(unsigned));
        if (e2 == cudaSuccess) e2 = cudaMalloc((void**)&ctx->pipes[k].retry_counts, RT_MAX_RETRIES * sizeof(unsigned));
        if (e2 == cudaSuccess) e2 = cudaHostAlloc((void**)&ctx->pipes[k].seen_counts, RT_SEEN_ROUNDS * sizeof(unsigned), cudaHostAllocDefault);
        if (e2 == cudaSuccess) memset(ctx->pipes[k].seen_counts, 0, RT_SEEN_ROUNDS * sizeof(unsigned));
        if (e2 == cudaSuccess) e2 = cudaHostAlloc((void**)&ctx->pipes[k].seen_retry, RT_MAX_RETRIES * sizeof(unsigned), cudaHostAllocDefault);
        if (e2 == cudaSuccess) for (int j = 0; j < RT_MAX_RETRIES; j++) ctx->pipes[k].seen_retry[j] = 0xffffffffu;      // unknown: full grids
        memset(&ctx->pipes[k].pool, 0, sizeof(PathPool));
    }
    if (e2 == cudaSuccess) e2 = cudaMemsetAsync(ctx->counters, 0, sizeof(rt_counters), ctx->stream);
    if (e2 != cudaSuccess)
    {
        std::string msg = std::string("context setup: ") + cudaGetErrorString(e2);
        delete ctx;
        return fail(nullptr, RT_ERR_CUDA, msg);
    }
    tuning_from_env(ctx);
    *out_ctx = ctx;
    return RT_OK;
}

int rt_gpu_destroy(rt_gpu_ctx* ctx)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_OK;
        cudaSetDevice(ctx->device);
        sync_all_streams(ctx);
        free_scene(ctx);
        free_frame(ctx);
        for (int k = 0; k < RT_FRAME_SLOTS; k++)
        {
            if (k == ctx->slot) continue;
            rt_gpu_ctx::FrameSlot& f = ctx->parked[k];
            cudaFree(f.accum); cudaFree(f.display); cudaFree(f.prim_ids); cudaFree(f.prim_dist); cudaFree(f.preview);
            if (f.ev0) cudaEventDestroy(f.ev0);
            if (f.ev1) cudaEventDestroy(f.ev1);
            if (f.stream) cudaStreamDestroy(f.stream);
        }
        cudaFree(ctx->counters);
        for (int k = 0; k < RT_PIPES; k++)
        {
            rt_gpu_ctx::Pipe& pp = ctx->pipes[k];
            if (pp.stream) cudaStreamSynchronize(pp.stream);
            for (void* q : pp.allocs) cudaFree(q);
            if (pp.seen_counts) cudaFreeHost(pp.seen_counts);
        if (pp.seen_retry) cudaFreeHost((void*)pp.seen_retry);
        cudaFree(pp.round_counters); cudaFree(pp.retry_counts); cudaFree(pp.retry[0]); cudaFree(pp.retry[1]); cudaFree(pp.samples);
            if (pp.done) cudaEventDestroy(pp.done);
            if (pp.stream) cudaStreamDestroy(pp.stream);
        }
        if (ctx->fork) cudaEventDestroy(ctx->fork);
        for (rt_gpu_ctx::TileTable& tt : ctx->tile_tables) cudaFree(tt.offsets);
        cudaFree(ctx->gather_staging);
        if (ctx->ev0) cudaEventDestroy(ctx->ev0);
        if (ctx->ev1) cudaEventDestroy(ctx->ev1);
        for (cudaEvent_t e : ctx->kev) cudaEventDestroy(e);
        for (cudaEvent_t e : ctx->cev) cudaEventDestroy(e);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return RT_OK;
    });
}

const char* rt_gpu_last_error(rt_gpu_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int rt_gpu_upload_scene(rt_gpu_ctx* ctx, const rt_scene_desc* s)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!s) return fail(ctx, RT_ERR_INVALID, "scene is null");
        if (s->abi_version != RT_GPU_ABI_VERSION) return fail(ctx, RT_ERR_INVALID, "rt_scene_desc.abi_version mismatch");
        if (s->num_shapes < 0 || s->num_materials < 0 || s->num_meshes < 0 || s->num_lights < 0)
            return fail(ctx, RT_ERR_INVALID, "negative count in scene");
        // validate indices before anything is copied
        bool needs_table = false;
        for (int i = 0; i < s->num_materials; i++)
        {
            const rt_material& m = s->materials[i];
            if (m.type < RT_MAT_DIFFUSE || m.type > RT_MAT_NULL) return fail(ctx, RT_ERR_INVALID, "unknown material type");
            if (m.type == RT_MAT_BLEND || m.type == RT_MAT_COMBINE)
                if (m.child_a < 0 || m.child_a >= s->num_materials || m.child_b < 0 || m.child_b >= s->num_materials)
                    return fail(ctx, RT_ERR_INVALID, "material child index out of range");
            if (m.type == RT_MAT_DIFFUSE || m.type == RT_MAT_CHECKER) needs_table = true;
        }
        for (int i = 0; i < s->num_shapes; i++)
        {
            const rt_shape& sh = s->shapes[i];
            if (sh.type < RT_SHAPE_SPHERE || sh.type > RT_SHAPE_TRIANGLE) return fail(ctx, RT_ERR_INVALID, "unknown shape type");
            if (sh.material >= s->num_materials) return fail(ctx, RT_ERR_INVALID, "shape material index out of range");
            if (sh.type == RT_SHAPE_MESH && (sh.mesh < 0 || sh.mesh >= s->num_meshes)) return fail(ctx, RT_ERR_INVALID, "shape mesh index out of range");
        }
        for (int i = 0; i < s->num_meshes; i++)
        {
            const rt_mesh& m = s->meshes[i];
            if (m.num_nodes < 0 || m.num_tris < 0 || m.num_textures < 0) return fail(ctx, RT_ERR_INVALID, "negative count in mesh");
            if (m.num_nodes > 0 && (!m.nodes || !m.tris || !m.shade)) return fail(ctx, RT_ERR_INVALID, "mesh arrays missing");
            if (m.num_textures > 0 && !m.textures) return fail(ctx, RT_ERR_INVALID, "mesh textures array missing");
            // first every index field on its own, then the nesting (which follows escape links)
            for (int k = 0; k < m.num_nodes; k++)
            {
                const rt_bvh_node& nd = m.nodes[k];
                if (nd.escape <= k || nd.escape > m.num_nodes || nd.tri >= m.num_tris)
                    return fail(ctx, RT_ERR_INVALID, "malformed BVH node (escape/tri index)");
            }
            for (int k = 0; k < m.num_nodes; k++)
            {
                const rt_bvh_node& nd = m.nodes[k];
                if (nd.tri < 0)
                {
                    // an inner node's range [k, escape) is its left subtree [k+1, r) followed by its right one [r, escape)
                    if (k + 1 >= nd.escape) return fail(ctx, RT_ERR_INVALID, "malformed BVH node (inner node without children)");
                    const int r = m.nodes[k + 1].escape;
                    if (r > nd.escape || (r < nd.escape && m.nodes[r].escape != nd.escape))
                        return fail(ctx, RT_ERR_INVALID, "malformed BVH node (subtrees do not nest)");
                }
                else if (nd.escape != k + 1) return fail(ctx, RT_ERR_INVALID, "malformed BVH node (leaf with a subtree)");
            }
            for (int k = 0; k < m.num_tris; k++)
            {
                if (m.tris[k].index < 0 || m.tris[k].index >= m.num_tris) return fail(ctx, RT_ERR_INVALID, "triangle index out of range");
                if (m.shade[k].texture >= m.num_textures) return fail(ctx, RT_ERR_INVALID, "texture index out of range");
            }
            for (int k = 0; k < m.num_textures; k++)
            {
                const rt_texture& t = m.textures[k];
                if (!texture_has_pixels(t)) continue;
                if (t.width <= 0 || t.height <= 0) return fail(ctx, RT_ERR_INVALID, "texture with non-positive size");
                if (!t.rgba && ((t.channels != 3 && t.channels != 4) || !t.lut))
                    return fail(ctx, RT_ERR_INVALID, "8-bit texture needs 3 or 4 channels and a 512-entry table");
            }
        }

        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(sync_all_streams(ctx));
        free_scene(ctx);

        DevScene d;
        memset(&d, 0, sizeof d);
        int rc;
        rt_shape* dshapes; rt_material* dmats; rt_light* dlights;
        if ((rc = upload(ctx, s->shapes, (size_t)s->num_shapes, &dshapes)) != RT_OK) return rc;
        if ((rc = upload(ctx, s->materials, (size_t)s->num_materials, &dmats)) != RT_OK) return rc;
        if ((rc = upload(ctx, s->lights, (size_t)s->num_lights, &dlights)) != RT_OK) return rc;
        d.shapes = dshapes; d.materials = dmats; d.lights = dlights;
        d.num_shapes = s->num_shapes; d.num_materials = s->num_materials; d.num_lights = s->num_lights;
        d.num_meshes = s->num_meshes;

        // ---- texture atlas: shelf-pack every decoded texture of the scene into one float4 cudaArray ----
        // device copies of 8-bit texels wait here until the expansion kernels have run
        struct TempGuard
        {
            std::vector<void*> v; cudaSurfaceObject_t* surf;
            ~TempGuard() { for (void* q : v) cudaFree(q); if (*surf) cudaDestroySurfaceObject(*surf); }
        };
        cudaSurfaceObject_t atlas_surface = 0;
        TempGuard temp_guard = { {}, &atlas_surface };
        std::vector<void*>& texel_temps = temp_guard.v;
        ctx->texel_upload_bytes = 0;
        struct AtlasRect { int x, y, w, h; };
        std::vector<AtlasRect> atlas_rects;          // in (mesh, slot) order, textured slots only
        size_t atlas_next = 0;
        cudaArray_t atlas_array = nullptr;
        {
            int max_w = 0;
            for (int i = 0; i < s->num_meshes; i++)
                for (int k = 0; k < s->meshes[i].num_textures; k++)
                    if (texture_has_pixels(s->meshes[i].textures[k]))
                    {
                        const rt_texture& t = s->meshes[i].textures[k];
                        atlas_rects.push_back(AtlasRect{ 0, 0, t.width, t.height });
                        if (t.width > max_w) max_w = t.width;
                    }
            if (!atlas_rects.empty())
            {
                const int shelf_w = max_w > 8192 ? max_w : 8192;
                std::vector<size_t> order(atlas_rects.size());
                for (size_t k = 0; k < order.size(); k++) order[k] = k;
                std::stable_sort(order.begin(), order.end(), [&](size_t l, size_t r) { return atlas_rects[l].h > atlas_rects[r].h; });
                int cx = 0, cy = 0, shelf_h = 0, used_w = 0;
                for (size_t k : order)
                {
                    AtlasRect& r = atlas_rects[k];
                    if (cx + r.w > shelf_w) { cy += shelf_h; cx = 0; shelf_h = 0; }
                    r.x = cx; r.y = cy;
                    cx += r.w;
                    if (r.h > shelf_h) shelf_h = r.h;
                    if (cx > used_w) used_w = cx;
                }
                const int atlas_h = cy + shelf_h;
                if (used_w > 131072 || atlas_h > 65536) return fail(ctx, RT_ERR_INVALID, "textures do not fit one atlas (131072 x 65536 texels)");
                cudaChannelFormatDesc fmt = cudaCreateChannelDesc<float4>();
                RT_CUDA(cudaMallocArray(&atlas_array, &fmt, (size_t)used_w, (size_t)atlas_h, cudaArraySurfaceLoadStore));
                ctx->arrays.push_back(atlas_array);
                ctx->scene_bytes += (size_t)used_w * atlas_h * 16;
                cudaResourceDesc res; memset(&res, 0, sizeof res);
                res.resType = cudaResourceTypeArray; res.res.array.array = atlas_array;
                cudaTextureDesc td; memset(&td, 0, sizeof td);
                td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
                td.filterMode = cudaFilterModePoint;       // texels only; RTexture::Sample's lerps are done in fp32 by hand
                td.readMode = cudaReadModeElementType;
                td.normalizedCoords = 0;
                cudaTextureObject_t obj = 0;
                RT_CUDA(cudaCreateTextureObject(&obj, &res, &td, nullptr));
                ctx->texobjs.push_back(obj);
                d.atlas = obj;
            }
        }

        std::vector<DevMesh> meshes((size_t)s->num_meshes);
        for (int i = 0; i < s->num_meshes; i++)
        {
            const rt_mesh& m = s->meshes[i];
            DevMesh& dm = meshes[i];
            memset(&dm, 0, sizeof dm);
            rt_bvh_node* dn; rt_tri* dt; rt_shade* dsh;
            if ((rc = upload(ctx, m.nodes, (size_t)m.num_nodes, &dn)) != RT_OK) return rc;
            if ((rc = upload(ctx, m.tris, (size_t)m.num_tris, &dt)) != RT_OK) return rc;
            if ((rc = upload(ctx, m.shade, (size_t)m.num_tris, &dsh)) != RT_OK) return rc;
            if (m.num_tris > 0)
            {
                // the device keeps the shading records in LEAF order (record k belongs to leaf triangle k): a hit then
                // fetches its triangle and its shading record side by side instead of one after the other
                rt_shade* leaf_order = nullptr;
                RT_CUDA(cudaMalloc((void**)&leaf_order, (size_t)m.num_tris * sizeof(rt_shade)));
                rt_shade_leaf_order_kernel<<<(unsigned)((m.num_tris + 255) / 256), 256, 0, ctx->stream>>>((const float4*)dt, (const float4*)dsh, (float4*)leaf_order, m.num_tris);
                RT_CUDA(cudaGetLastError());
                ctx->launches++;
                ctx->scene_allocs.push_back(leaf_order);
                texel_temps.push_back(dsh);             // freed once the stream has drained (end of this call)
                ctx->scene_allocs.erase(std::find(ctx->scene_allocs.begin(), ctx->scene_allocs.end(), (void*)dsh));
                dsh = leaf_order;
            }
            if (m.num_nodes > 0)
            {
                rt_patch_right_child<<<(unsigned)((m.num_nodes + 255) / 256), 256, 0, ctx->stream>>>(dn, m.num_nodes);
                RT_CUDA(cudaGetLastError());
            }
            dm.nodes = (const float4*)dn; dm.tris = (const float4*)dt; dm.shade = (const float4*)dsh;
            dm.octo = nullptr;
            if (m.num_nodes > 0 && ctx->tune_octo)
            {
                std::vector<rt_bvh_node> octo;
                build_octo(m.nodes, m.num_nodes, octo);
                if (octo.size() / 8 < (1u << 24))
                {
                    rt_bvh_node* docto = nullptr;
                    if ((rc = upload(ctx, octo.data(), octo.size(), &docto)) != RT_OK) return rc;
                    RT_CUDA(cudaStreamSynchronize(ctx->stream));       // octo is a local
                    dm.octo = (const float4*)docto;
                }
            }
            dm.num_nodes = m.num_nodes; dm.num_tris = m.num_tris; dm.num_textures = m.num_textures;
            float scale = 0.0f;
            if (m.num_nodes > 0)
                for (int k = 0; k < 3; k++)
                {
                    scale = fmaxf(scale, fabsf(m.nodes[0].bmin[k]));
                    scale = fmaxf(scale, fabsf(m.nodes[0].bmax[k]));
                }
            dm.cull_scale = scale;
            std::vector<DevTexture> texs((size_t)m.num_textures);
            for (int k = 0; k < m.num_textures; k++)
            {
                const rt_texture& t = m.textures[k];
                DevTexture& dt2 = texs[k];
                dt2.x0 = dt2.y0 = 0; dt2.width = t.width; dt2.height = t.height;
                if (!texture_has_pixels(t)) { dt2.width = dt2.height = 0; continue; }
                const AtlasRect& rc2 = atlas_rects[atlas_next++];
                dt2.x0 = rc2.x; dt2.y0 = rc2.y;
                if (t.rgba)
                    RT_CUDA(cudaMemcpy2DToArrayAsync(atlas_array, (size_t)rc2.x * 16, (size_t)rc2.y, t.rgba, (size_t)t.width * 16,
                                                     (size_t)t.width * 16, (size_t)t.height, cudaMemcpyHostToDevice, ctx->stream));
                else
                {
                    // 8-bit texels + the host's 256-entry powf table travel (3-4 B per texel instead of 16); the float4
                    // texels of Texture.cpp:119-151 are produced here, bit-identical by construction (table lookups only)
                    const size_t count = (size_t)t.width * t.height;
                    uint8_t* d8 = nullptr; float* dlut = nullptr;
                    RT_CUDA(cudaMalloc((void**)&d8, count * (size_t)t.channels));
                    texel_temps.push_back(d8);
                    RT_CUDA(cudaMalloc((void**)&dlut, 512 * sizeof(float)));
                    texel_temps.push_back(dlut);
                    RT_CUDA(cudaMemcpyAsync(d8, t.texels8, count * (size_t)t.channels, cudaMemcpyHostToDevice, ctx->stream));
                    RT_CUDA(cudaMemcpyAsync(dlut, t.lut, 512 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
                    if (!atlas_surface)
                    {
                        cudaResourceDesc sres; memset(&sres, 0, sizeof sres);
                        sres.resType = cudaResourceTypeArray; sres.res.array.array = atlas_array;
                        RT_CUDA(cudaCreateSurfaceObject(&atlas_surface, &sres));
                    }
                    const dim3 grid((unsigned)((t.width + 31) / 32), (unsigned)((t.height + 7) / 8));
                    rt_expand_texels_kernel<<<grid, dim3(32, 8), 0, ctx->stream>>>(atlas_surface, d8, dlut, t.width, t.height, t.channels, rc2.x, rc2.y);
                    RT_CUDA(cudaGetLastError());
                    ctx->launches++;
                    ctx->texel_upload_bytes += count * (size_t)t.channels + 512 * sizeof(float);
                }
                if (t.rgba) ctx->texel_upload_bytes += (size_t)t.width * t.height * 16;
                ctx->host_textures.push_back(dt2);
            }
            // a shade record may only name a slot that holds pixels
            for (int k = 0; k < m.num_tris; k++)
                if (m.shade[k].texture >= 0 && !texture_has_pixels(m.textures[m.shade[k].texture]))
                    return fail(ctx, RT_ERR_INVALID, "shade record names an empty texture slot");
            DevTexture* dtex;
            if ((rc = upload(ctx, texs.data(), texs.size(), &dtex)) != RT_OK) return rc;
            dm.textures = dtex;
            RT_CUDA(cudaStreamSynchronize(ctx->stream));   // texs is a local
        }
        DevMesh* dmeshes;
        if ((rc = upload(ctx, meshes.data(), meshes.size(), &dmeshes)) != RT_OK) return rc;
        d.meshes = dmeshes;
        std::vector<int> top_tags(RT_TOP_SLOTS, -1);
        std::vector<rt_bvh_node> top_nodes(RT_TOP_SLOTS);
        if (s->num_meshes > 0 && s->meshes[0].num_nodes > 0)
        {
            // the shallowest levels of mesh 0, breadth first, into hashed slots (a taken slot stays with the shallower
            // node); children of node k: k + 1 and the escape of k + 1.  The device copy keeps the right child in `tri`.
            const rt_mesh& m0 = s->meshes[0];
            std::vector<int> level(1, 0), next_level;
            int placed = 0;
            while (!level.empty() && placed < RT_TOP_SLOTS * 3 / 4)
            {
                next_level.clear();
                for (int k : level)
                {
                    const unsigned slot = top_slot(k);
                    if (top_tags[slot] < 0)
                    {
                        top_tags[slot] = k; top_nodes[slot] = m0.nodes[k]; placed++;
                        if (m0.nodes[k].tri < 0) top_nodes[slot].tri = -2 - (k + 1 < m0.num_nodes ? m0.nodes[k + 1].escape : m0.num_nodes);
                    }
                    if (m0.nodes[k].tri < 0)
                    {
                        next_level.push_back(k + 1);
                        const int right = m0.nodes[k + 1].escape;
                        if (right < m0.nodes[k].escape) next_level.push_back(right);
                    }
                }
                level.swap(next_level);
            }
            int* dtags; rt_bvh_node* dtop;
            if ((rc = upload(ctx, top_tags.data(), top_tags.size(), &dtags)) != RT_OK) return rc;
            if ((rc = upload(ctx, top_nodes.data(), top_nodes.size(), &dtop)) != RT_OK) return rc;
            d.top_tags = dtags; d.top_nodes = (const float4*)dtop; d.top_of = meshes[0].nodes;
        }

        if (s->num_unit_vectors > 0 && s->unit_vectors)
        {
            // pad xyz -> float4 so one 16-byte load fetches a direction
            const size_t n = s->num_unit_vectors;
            float4* dv = nullptr;
            RT_CUDA(cudaMalloc((void**)&dv, n * sizeof(float4)));
            ctx->scene_allocs.push_back(dv);
            ctx->scene_bytes += n * sizeof(float4);
            // (copies on the context's stream: a blocking cudaMemcpy from pageable memory is not ordered against the
            // non-blocking streams this context renders on)
            const size_t step = 1u << 20;
            std::vector<float4> stage[2];
            stage[0].resize(step < n ? step : n); stage[1].resize(step < n ? step : n);
            cudaEvent_t staged[2] = { nullptr, nullptr };
            RT_CUDA(cudaEventCreateWithFlags(&staged[0], cudaEventDisableTiming));
            RT_CUDA(cudaEventCreateWithFlags(&staged[1], cudaEventDisableTiming));
            cudaError_t ue = cudaSuccess;
            int turn = 0;
            for (size_t lo = 0; lo < n && ue == cudaSuccess; lo += step, turn ^= 1)
            {
                const size_t cnt = (n - lo) < step ? (n - lo) : step;
                if (lo >= 2 * step) ue = cudaEventSynchronize(staged[turn]);        // the copy that last read this buffer
                float4* st = stage[turn].data();
                for (size_t k = 0; k < cnt; k++)
                {
                    const float* v = s->unit_vectors + 3 * (lo + k);
                    st[k] = make_float4(v[0], v[1], v[2], 0.0f);
                }
                if (ue == cudaSuccess) ue = cudaMemcpyAsync(dv + lo, st, cnt * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream);
                if (ue == cudaSuccess) ue = cudaEventRecord(staged[turn], ctx->stream);
            }
            if (ue == cudaSuccess) ue = cudaStreamSynchronize(ctx->stream);
            cudaEventDestroy(staged[0]); cudaEventDestroy(staged[1]);
            RT_CUDA(ue);
            d.unit_vectors = dv;
            d.num_unit_vectors = s->num_unit_vectors;
        }
        for (int k = 0; k < 3; k++) d.eye[k] = s->eye[k];
        d.dir_z = s->dir_z; d.ray_distance = s->ray_distance; d.bounce_offset = s->bounce_offset;
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->scene = d;
        ctx->has_scene = true;
        ctx->needs_table = needs_table;
        ctx->host_shape_is_mesh.assign((size_t)s->num_shapes, 0);
        for (int i = 0; i < s->num_shapes; i++) ctx->host_shape_is_mesh[i] = s->shapes[i].type == RT_SHAPE_MESH ? 1 : 0;
        ctx->all_bounded = true;
        for (int i = 0; i < s->num_shapes; i++) if (!s->shapes[i].has_bounds) ctx->all_bounded = false;
        return RT_OK;
    });
}

int rt_gpu_set_frame_slot(rt_gpu_ctx* ctx, int32_t slot)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (slot < 0 || slot >= RT_FRAME_SLOTS) return fail(ctx, RT_ERR_INVALID, "frame slot out of range");
        ctx->slots_used = true;
        if (!(ctx->slot_mask & (1u << slot))) { ctx->slot_mask |= 1u << slot; ctx->slots_touched++; }
        if (slot == ctx->slot) return RT_OK;
        RT_CUDA(cudaSetDevice(ctx->device));
        rt_gpu_ctx::FrameSlot& in = ctx->parked[slot];
        if (!in.stream)
        {
            RT_CUDA(cudaStreamCreateWithFlags(&in.stream, cudaStreamNonBlocking));
            RT_CUDA(cudaEventCreate(&in.ev0));
            RT_CUDA(cudaEventCreate(&in.ev1));
        }
        park_slot(ctx, ctx->parked[ctx->slot]);
        unpark_slot(ctx, in);
        in = rt_gpu_ctx::FrameSlot();
        ctx->slot = slot;
        return RT_OK;
    });
}

int rt_gpu_get_frame_slot(rt_gpu_ctx* ctx) { return ctx ? ctx->slot : -1; }

int rt_gpu_reset_accum(rt_gpu_ctx* ctx, int32_t width, int32_t height)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (width <= 0 || height <= 0 || (long long)width * height > 0x7fffffffLL) return fail(ctx, RT_ERR_INVALID, "bad frame size");
        RT_CUDA(cudaSetDevice(ctx->device));
        const size_t n = (size_t)width * height;
        if (width != ctx->width || height != ctx->height)
        {
            RT_CUDA(cudaStreamSynchronize(ctx->stream));
            free_frame(ctx);
            RT_CUDA(cudaMalloc((void**)&ctx->accum, n * sizeof(float4)));
            RT_CUDA(cudaMalloc((void**)&ctx->display, n * sizeof(uint32_t)));
            RT_CUDA(cudaMalloc((void**)&ctx->prim_ids, n * sizeof(int2)));
            RT_CUDA(cudaMalloc((void**)&ctx->prim_dist, n * sizeof(float)));
            ctx->width = width; ctx->height = height;
        }
        RT_CUDA(cudaMemsetAsync(ctx->accum, 0, n * sizeof(float4), ctx->stream));
        RT_CUDA(cudaMemsetAsync(ctx->display, 0, n * sizeof(uint32_t), ctx->stream));
        RT_CUDA(cudaMemsetAsync(ctx->prim_ids, 0xff, n * sizeof(int2), ctx->stream));
        RT_CUDA(cudaMemsetAsync(ctx->prim_dist, 0, n * sizeof(float), ctx->stream));
        return RT_OK;
    });
}

int rt_gpu_render_tile(rt_gpu_ctx* ctx, const rt_render_params* p)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!p) return fail(ctx, RT_ERR_INVALID, "params is null");
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_render_tile before rt_gpu_upload_scene");
        if (p->width <= 0 || p->height <= 0 || (long long)p->width * p->height > 0x7fffffffLL) return fail(ctx, RT_ERR_INVALID, "bad frame size");
        const int npix = p->width * p->height;
        if (p->start < 0 || p->end >= npix) return fail(ctx, RT_ERR_INVALID, "pixel range outside the frame");
        if (p->mode < RT_MODE_PATH || p->mode > RT_MODE_PRIMARY) return fail(ctx, RT_ERR_INVALID, "unknown mode");
        if (p->traverse != RT_TRAVERSE_EXACT && p->traverse != RT_TRAVERSE_CULLED) return fail(ctx, RT_ERR_INVALID, "unknown traverse");
        if (p->mode == RT_MODE_PATH && ctx->needs_table && ctx->scene.num_unit_vectors == 0)
            return fail(ctx, RT_ERR_INVALID, "scene has Diffuse materials but no unit-vector table (rt_host_set_unit_vectors)");
        if (p->max_bounce < 0 || p->max_bounce > RT_MAX_PATH_DEPTH) return fail(ctx, RT_ERR_INVALID, "max_bounce must be in [0, 32]");
        if (p->pass_count < 0 || p->pass_begin < 0) return fail(ctx, RT_ERR_INVALID, "negative pass range");
        if (p->tile_count > 1 && (p->tile_size <= 0 || p->tile_rank < 0 || p->tile_rank >= p->tile_count))
            return fail(ctx, RT_ERR_INVALID, "bad tile ownership fields");
        RT_CUDA(cudaSetDevice(ctx->device));
        if (p->width != ctx->width || p->height != ctx->height)
        {
            int rc = rt_gpu_reset_accum(ctx, p->width, p->height);
            if (rc != RT_OK) return rc;
        }
        RT_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
        ctx->timed = true;
        ctx->kev_used = 0;
        ctx->cev_used = 0;
        // rt_gpu_time_kernels(ctx, 2): an event before every launch, tagged with the kernel's class; the time to
        // the next event is that launch's (meaningful with one pipe: launches then follow each other on one stream)
        auto mark = [&](int cls, cudaStream_t st) -> cudaError_t {
            if (!ctx->time_classes) return cudaSuccess;
            if ((int)ctx->cev.size() <= ctx->cev_used)
            {
                cudaEvent_t e = nullptr;
                const cudaError_t ce = cudaEventCreate(&e);
                if (ce != cudaSuccess) return ce;
                ctx->cev.push_back(e); ctx->cev_cls.push_back(-1);
            }
            ctx->cev_cls[ctx->cev_used] = cls;
            return cudaEventRecord(ctx->cev[ctx->cev_used++], st);
        };
        if (p->end < p->start || (p->mode != RT_MODE_PRIMARY && p->pass_count == 0))
        {
            RT_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
            return RT_OK;                                 // empty task
        }

        RenderArgs a;
        memset(&a, 0, sizeof a);
        a.width = p->width; a.height = p->height; a.start = p->start; a.end = p->end;
        a.mode = p->mode; a.max_bounce = p->max_bounce; a.antialias = p->antialias ? 1 : 0; a.seed = p->seed;
        a.spp = (a.antialias && p->mode != RT_MODE_PRIMARY) ? 4 : 1;
        if (p->mode == RT_MODE_PRIMARY) a.antialias = 0;
        a.tiled = (p->tile_count > 1 && p->tile_size > 0) ? 1 : 0;
        a.tile_size = p->tile_size; a.tile_count = p->tile_count; a.tile_rank = p->tile_rank;
        if (a.tiled)
        {
            a.tiles_x = (p->width + p->tile_size - 1) / p->tile_size;
            const int tiles_y = (p->height + p->tile_size - 1) / p->tile_size;
            const int ntiles = a.tiles_x * tiles_y;
            const int owned = p->tile_rank < ntiles ? (ntiles - p->tile_rank + p->tile_count - 1) / p->tile_count : 0;
            a.blocks_x = (p->tile_size + 7) / 8;
            a.blocks_per_tile = a.blocks_x * ((p->tile_size + 3) / 4);
            a.num_blocks = (unsigned)owned * (unsigned)a.blocks_per_tile;
        }
        else
        {
            a.row0 = p->start / p->width;
            a.rows = p->end / p->width - a.row0 + 1;
            a.blocks_x = (p->width + 7) / 8;
            a.blocks_per_tile = a.blocks_x * ((a.rows + 3) / 4);
            a.num_blocks = (unsigned)a.blocks_per_tile;
        }
        if (p->mode == RT_MODE_PREVIEW && !ctx->preview)
        {
            RT_CUDA(cudaMalloc((void**)&ctx->preview, (size_t)npix * sizeof(float4)));
            RT_CUDA(cudaMemsetAsync(ctx->preview, 0, (size_t)npix * sizeof(float4), ctx->stream));
        }
        a.accum = ctx->accum; a.display = ctx->display; a.prim_ids = ctx->prim_ids; a.prim_dist = ctx->prim_dist;
        a.preview = ctx->preview;
        a.counters = ctx->counters;
        a.exact = p->traverse == RT_TRAVERSE_EXACT ? 1 : 0;
        a.all_bounded = ctx->all_bounded ? 1 : 0;
        if (a.num_blocks == 0)
        {
            RT_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
            return RT_OK;
        }

        int rc = init_walk_grid(ctx);
        if (rc != RT_OK) return rc;
        // rounds: one mesh walk per round; a path needs at most (segments) x (mesh shapes) walks
        int mesh_shapes = 0;
        for (int i = 0; i < ctx->scene.num_shapes; i++) mesh_shapes += ctx->host_shape_is_mesh[i] ? 1 : 0;
        const int segments = p->mode == RT_MODE_PATH ? (p->max_bounce > 0 ? p->max_bounce : 1)
                           : p->mode == RT_MODE_WHITTED ? 1 + ctx->scene.num_lights : 1;
        const int rounds = segments * (mesh_shapes > 0 ? mesh_shapes : 1);
        if (rounds >= RT_MAX_ROUNDS) return fail(ctx, RT_ERR_INVALID, "max_bounce x mesh shapes exceeds the round table");

        const int total_passes = p->mode == RT_MODE_PRIMARY ? 1 : p->pass_count;
        // sample buffer: whole frames of float4 per sample; split long calls into pass chunks
        // A call with fewer camera rays (one rank's share of a multi-GPU frame) is split in fewer, longer chunks:
        // every chunk pays its thin last rounds once, and there is less dense work to hide them behind.
        const unsigned long long call_items = (unsigned long long)a.num_blocks * 32ull * (unsigned long long)a.spp * (unsigned long long)total_passes;
        const size_t sample_budget = ctx->tune_sample_budget ? ctx->tune_sample_budget
                                   : call_items < RT_FEW_ITEMS ? RT_SAMPLE_BUDGET_FEW_BYTES : RT_SAMPLE_BUDGET_BYTES;
        size_t passes_per_chunk = sample_budget / ((size_t)npix * sizeof(float4) * (size_t)a.spp);
        // ... unless frames overlap each other (frame slots): then one chunk, whose tail the NEXT frames cover
        const int few_chunks = ctx->tune_few_chunks > 0 ? ctx->tune_few_chunks : (ctx->slots_used ? 1 : 2);
        if (!ctx->tune_sample_budget && call_items < RT_FEW_ITEMS && few_chunks > 1 &&
            passes_per_chunk > ((size_t)total_passes + few_chunks - 1) / few_chunks)
            passes_per_chunk = ((size_t)total_passes + few_chunks - 1) / few_chunks;     // equal chunks (their pipes overlap)
        if (passes_per_chunk < 1) passes_per_chunk = 1;
        if (passes_per_chunk > (size_t)total_passes) passes_per_chunk = (size_t)total_passes;
        {
            // the work list of one launch is indexed with 32 bits
            const unsigned long long per_pass = (unsigned long long)a.num_blocks * 32ull * (unsigned long long)a.spp;
            if (per_pass > 0xffffffffull) return fail(ctx, RT_ERR_INVALID, "frame too large for one launch");
            const size_t fit = (size_t)(0xffffffffull / per_pass);
            if (passes_per_chunk > fit) passes_per_chunk = fit;
        }
        {
            // equal-sized chunks (16 passes with room for 5 -> 4 x 4, not 5+5+5+1)
            const size_t nchunks = ((size_t)total_passes + passes_per_chunk - 1) / passes_per_chunk;
            passes_per_chunk = ((size_t)total_passes + nchunks - 1) / nchunks;
        }
        const int nchunks_total = (int)(((size_t)total_passes + passes_per_chunk - 1) / passes_per_chunk);
        if (p->mode != RT_MODE_PRIMARY)
        {
            const size_t need = passes_per_chunk * (size_t)a.spp * (size_t)npix;
            for (int k = 0; k < RT_PIPES && (k < nchunks_total || ctx->slots_used); k++)
            {
                rt_gpu_ctx::Pipe& pp = ctx->pipes[k];
                if (k >= ctx->tune_pipes) break;
                if (need > pp.samples_cap)
                {
                    RT_CUDA(sync_all_streams(ctx));
                    cudaFree(pp.samples); pp.samples = nullptr; pp.samples_cap = 0;
                    RT_CUDA(cudaMalloc((void**)&pp.samples, need * sizeof(float4)));
                    pp.samples_cap = need;
                }
            }
        }

        // ---- batches, pools and pipes ------------------------------------------------------------------------
        // A batch is as large as possible (every batch pays the latency of its thin last rounds once); its
        // pool is smaller: most camera rays never become paths.  When a pool does fill up, the items it
        // turned away are generated again by retry passes.
        const unsigned long long items_per_chunk = (unsigned long long)passes_per_chunk * a.spp * a.num_blocks * 32ull;
        const int npipes = ctx->tune_pipes;
        const size_t batch = (size_t)((items_per_chunk + 255ull) & ~255ull);
        const size_t levels = p->mode == RT_MODE_PATH ? (size_t)(p->max_bounce > 0 ? p->max_bounce : 1) : 1;
        const bool whitted = p->mode == RT_MODE_WHITTED;
        size_t pool_want = 0;
        if ((rc = plan_pools(ctx, batch, levels, whitted, &pool_want)) != RT_OK) return rc;
        const int retries = (int)((batch + pool_want - 1) / pool_want) - 1;
        if (retries >= RT_MAX_RETRIES) return fail(ctx, RT_ERR_NOMEM, "path pool too small for this frame (raise the pool size)");
        {
            if ((rc = grow_pools(ctx, pool_want, levels, whitted)) != RT_OK) return rc;
            for (int k = 0; k < RT_PIPES; k++)
            {
                rt_gpu_ctx::Pipe& pp = ctx->pipes[k];
                if (retries > 0 && batch > pp.retry_cap)
                {
                    RT_CUDA(cudaStreamSynchronize(ctx->stream));
                    RT_CUDA(cudaStreamSynchronize(pp.stream));
                    cudaFree(pp.retry[0]); cudaFree(pp.retry[1]); pp.retry[0] = pp.retry[1] = nullptr; pp.retry_cap = 0;
                    RT_CUDA(cudaMalloc((void**)&pp.retry[0], batch * 4));
                    RT_CUDA(cudaMalloc((void**)&pp.retry[1], batch * 4));
                    pp.retry_cap = batch;
                }
            }
        }
        const bool cull = p->traverse == RT_TRAVERSE_CULLED;
        // the round whose queue is still in camera order is walked as packets (bounce and shadow rays of later
        // rounds are not coherent enough: measured slower, see DESIGN.md)
        const int packet_rounds = ctx->tune_packet_rounds >= 0 ? ctx->tune_packet_rounds : 1;
        const unsigned walk_grid = (unsigned)(ctx->num_sms * ctx->walk_blocks_per_sm);

        // Chunks alternate between the pipes.  Each pipe renders into its own sample buffer and folds it
        // itself; the only cross-pipe order is fold(k) before fold(k+1) (AddPixel sums in pass order), so
        // the thin, latency-bound last rounds of chunk k overlap the dense first rounds of chunk k+1.
        RT_CUDA(cudaEventRecord(ctx->fork, ctx->stream));
        PipeGuard guard = { ctx, { false }, false };
        bool (&used)[RT_PIPES] = guard.used;
        int chunk_index = 0, last_pipe = -1;
        // With frame slots in use consecutive calls rotate through the pipes, so that the next frame's chunks do
        // not queue up behind this frame's thin last rounds on the same streams.
        const int pipe_base = ctx->slots_used ? ctx->pipe_cursor % npipes : 0;
        for (int done = 0; done < total_passes; done += (int)passes_per_chunk, chunk_index++)
        {
            const int chunk = (total_passes - done) < (int)passes_per_chunk ? (total_passes - done) : (int)passes_per_chunk;
            const int pipe = (pipe_base + chunk_index) % npipes;
            rt_gpu_ctx::Pipe& pp = ctx->pipes[pipe];
            if (!used[pipe]) { RT_CUDA(cudaStreamWaitEvent(pp.stream, ctx->fork, 0)); used[pipe] = true; }
            a.pass_begin = p->pass_begin + done;
            a.num_samples = chunk * a.spp;
            a.num_items = (unsigned)((unsigned long long)a.num_samples * a.num_blocks * 32ull);
            a.samples = pp.samples;
            {
                WaveArgs w = pipe_wave_args(ctx, pp, packet_rounds > 0 && mesh_shapes > 0 ? 1 : 0);
                w.item_begin = 0u;
                w.item_count = a.num_items;
                unsigned gen_grid = (a.num_blocks * 32u + 255u) / 256u;
                if (gen_grid > (unsigned)ctx->num_sms * 8u) gen_grid = (unsigned)ctx->num_sms * 8u;
                // the shade grid strides over the round's queue; a few waves are enough
                unsigned shade_grid = (unsigned)((ctx->pool_cap < w.item_count ? ctx->pool_cap : w.item_count) + 255u) / 256u;
                const unsigned shade_max = (unsigned)ctx->num_sms * 16u;
                if (shade_grid > shade_max) shade_grid = shade_max;
                if (retries > 0) RT_CUDA(cudaMemsetAsync(pp.retry_counts, 0, RT_MAX_RETRIES * sizeof(unsigned), pp.stream));
                // (the shape of a call for this purpose: mode and depth; chunks of a frame differ a little in size, which the
                // threshold does not care about)
                const unsigned long long signature = ((unsigned long long)p->mode << 8) ^ (unsigned long long)p->max_bounce ^ ((unsigned long long)(a.tiled ? a.tile_count : 1) << 16);
                // (a racy read of pinned memory the device may be updating: either batch's sizes will do)
                const volatile unsigned* seen_counts = (pp.seen_counts && pp.seen_signature == signature && pp.seen_counts[0] != 0u) ? pp.seen_counts : nullptr;
                for (int pass = 0; pass <= retries; pass++)
                {
                    // A retry pass that had (next to) nothing to do last time — the usual case: pools are sized so that
                    // retries are rare — is launched with one CTA per SM throughout: its ~40 launches would otherwise put
                    // ~35 000 CTAs on the machine only to find their queues empty.  If it does have work it is just slower.
                    const bool small_pass = pass > 0 && seen_counts && ctx->tune_thin_from_round == 0 && pp.seen_retry[pass - 1] < RT_SMALL_RETRY;
                    const unsigned sms = (unsigned)ctx->num_sms;
                    // pass 0 generates the slice; pass k > 0 the items pass k-1 could not place
                    w.retry_in = pass > 0 ? pp.retry[(pass - 1) & 1] : nullptr;
                    w.retry_in_count = pass > 0 ? pp.retry_counts + (pass - 1) : nullptr;
                    w.retry_out = retries > 0 ? pp.retry[pass & 1] : nullptr;
                    w.retry_out_count = retries > 0 ? pp.retry_counts + pass : nullptr;
                    RT_CUDA(mark(RT_KERNEL_OTHER, pp.stream));
                    RT_CUDA(cudaMemsetAsync(pp.round_counters, 0, (6 * RT_MAX_ROUNDS + 1) * sizeof(unsigned), pp.stream));
                    RT_CUDA(mark(RT_KERNEL_GENERATE, pp.stream));
                    RT_CUDA(cull ? launch_generate<true>(p->mode, small_pass ? sms : gen_grid, pp.stream, ctx->scene, a, w)
                                 : launch_generate<false>(p->mode, small_pass ? sms : gen_grid, pp.stream, ctx->scene, a, w));
                    ctx->launches++;
                    // (tooling: RT_FINISH_ROUND = k > 0 runs rounds >= k in the finishing kernel, -1 every round)
                    const int wave_rounds = ctx->tune_finish_round < 0 ? 0
                                          : (ctx->tune_finish_round > 0 && ctx->tune_finish_round < rounds) ? ctx->tune_finish_round : rounds;
                    for (int round = 0; round < wave_rounds; round++)
                    {
                        // Frames in flight: a late round holds a few thousand paths, yet its three launches would each
                        // put a full persistent grid in front of the dense kernels of the frames behind it.  The size
                        // of round r is known from the last batch this pipe rendered with the same shape (copied to
                        // pinned host memory when that batch ran; unknown -> full grids): a round that was small is
                        // launched with a quarter of the CTAs — once three or more frame slots are in use (with fewer frames
                        // in flight, or with a single pipe, a late round is exposed, and then it wants the full grid).  Grid sizes
                        // never change results.
                        const bool thin = ctx->tune_thin_from_round > 0 ? round >= ctx->tune_thin_from_round
                                        : (ctx->slots_touched >= 3 && npipes > 1 && ctx->tune_thin_from_round == 0 && seen_counts && round < RT_SEEN_ROUNDS &&
                                           seen_counts[round] < ctx->tune_thin_grid_count);
                        if ((rc = enqueue_round(ctx, pp, a, w, p->mode, round, cull, packet_rounds, mesh_shapes > 0, small_pass, thin,
                                                walk_grid, shade_grid, true, mark)) != RT_OK)
                            return rc;
                    }
                    if (pass == 0 && pp.seen_counts)
                    {
                        // this batch's round sizes, for the grids of the next batch on this pipe
                        RT_CUDA(cudaMemcpyAsync(pp.seen_counts, pp.round_counters, RT_SEEN_ROUNDS * sizeof(unsigned), cudaMemcpyDeviceToHost, pp.stream));
                        pp.seen_signature = signature;
                    }
                    if (wave_rounds < rounds)
                    {
                        // everything still alive after the wavefront rounds runs to its end in one launch
                        RT_CUDA(mark(RT_KERNEL_OTHER, pp.stream));
                        RT_CUDA(cull ? launch_finish<true>(p->mode, (unsigned)ctx->num_sms * 4u, pp.stream, ctx->scene, a, w, wave_rounds)
                                     : launch_finish<false>(p->mode, (unsigned)ctx->num_sms * 4u, pp.stream, ctx->scene, a, w, wave_rounds));
                        ctx->launches++;
                    }
                }
            }
            if (retries > 0 && pp.seen_retry)
                RT_CUDA(cudaMemcpyAsync((void*)pp.seen_retry, pp.retry_counts, RT_MAX_RETRIES * sizeof(unsigned), cudaMemcpyDeviceToHost, pp.stream));
            if (p->mode != RT_MODE_PRIMARY)
            {
                if (last_pipe >= 0 && last_pipe != pipe) RT_CUDA(cudaStreamWaitEvent(pp.stream, ctx->pipes[last_pipe].done, 0));
                const int n = p->end - p->start + 1;
                RT_CUDA(mark(RT_KERNEL_FOLD, pp.stream));
                rt_resolve_kernel<<<(n + 255) / 256, 256, 0, pp.stream>>>(a, chunk);
                RT_CUDA(cudaGetLastError());
                ctx->launches++;
            }
            RT_CUDA(mark(-1, pp.stream));
            RT_CUDA(cudaEventRecord(pp.done, pp.stream));
            last_pipe = pipe;
        }
        // join: the context stream continues after every pipe
        for (int k = 0; k < RT_PIPES; k++)
            if (used[k]) RT_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->pipes[k].done, 0));
        guard.joined = true;
        ctx->pipe_cursor = (pipe_base + chunk_index) % npipes;
        RT_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
        return RT_OK;
    });
}

// A batch of ray queries runs through the render's wavefront (enqueue_ray_batch): query generate, then one round per
// mesh a ray can reach, with the shade kernel in a query mode.
int rt_gpu_query_rays(rt_gpu_ctx* ctx, const rt_ray_query* q, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!q) return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: query is null");
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_query_rays before rt_gpu_upload_scene");
        if (q->n < 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: negative ray count");
        if (q->kind != RT_QUERY_NEAREST && q->kind != RT_QUERY_ANY) return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: unknown query kind");
        if (q->traverse != RT_TRAVERSE_EXACT && q->traverse != RT_TRAVERSE_CULLED) return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: unknown traverse");
        if (q->kind == RT_QUERY_ANY && (q->tri || q->hit))
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: tri and hit are results of RT_QUERY_NEAREST only");
        if (q->n == 0) return RT_OK;
        if (!q->rays || !q->shape) return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: rays and shape are required");
        RT_CUDA(cudaSetDevice(ctx->device));
        const void* ptrs[4] = { q->rays, q->shape, q->tri, q->hit };
        const char* names[4] = { "rays", "shape", "tri", "hit" };
        for (int k = 0; k < 4; k++)
            if (ptrs[k] && !on_device(ctx, ptrs[k]))
                return fail(ctx, RT_ERR_INVALID, std::string("rt_gpu_query_rays: ") + names[k] + " is not device memory of the context's GPU");
        int mesh_shapes = 0;
        for (int i = 0; i < ctx->scene.num_shapes; i++) mesh_shapes += ctx->host_shape_is_mesh[i] ? 1 : 0;
        const int rounds = mesh_shapes;                 // a query walks each mesh whose bounds it enters at most once
        if (rounds >= RT_MAX_ROUNDS) return fail(ctx, RT_ERR_INVALID, "rt_gpu_query_rays: mesh shapes exceed the round table");
        int rc = init_walk_grid(ctx);
        if (rc != RT_OK) return rc;
        const size_t n = (size_t)q->n;
        size_t pool_want = 0;
        if ((rc = plan_pools(ctx, (n + 255) & ~(size_t)255, 1, false, &pool_want)) != RT_OK) return rc;
        if ((rc = grow_pools(ctx, pool_want, 1, false)) != RT_OK) return rc;
        const size_t piece = pool_want & ~(size_t)31;   // path_alloc_packet takes 32 ids per warp with a live ray

        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        const bool cull = q->traverse == RT_TRAVERSE_CULLED;
        const int qmode = q->kind == RT_QUERY_ANY ? RT_QMODE_ANY : RT_QMODE_NEAREST;
        RenderArgs a;
        memset(&a, 0, sizeof a);
        a.mode = qmode;
        a.counters = ctx->counters;
        a.exact = cull ? 0 : 1;
        a.all_bounded = ctx->all_bounded ? 1 : 0;
        return enqueue_ray_batch(ctx, a, n, piece, qmode, rounds, mesh_shapes > 0, cull, st,
                                 [&](RenderArgs& pa, size_t begin, size_t) {
                                     pa.q_rays = q->rays + 7 * begin;
                                     pa.q_shape = q->shape + begin;
                                     pa.q_tri = q->tri ? q->tri + begin : nullptr;
                                     pa.q_hit = q->hit ? q->hit + 11 * begin : nullptr;
                                 });
    });
}

// Radiance of a batch of rays: the render's path (or preview / Whitted composition) from the caller's rays instead of
// the camera's.  The query generate kernel starts each path; the walk, long-walk and shade kernels run in the plain
// render mode, and the sample of ray i lands at rgba[i]: the piece's part of rgba is its sample buffer, one frame of
// `count` x 1 pixels, sample slot 0.
int rt_gpu_radiance_rays(rt_gpu_ctx* ctx, const rt_radiance_query* q, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!q) return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: query is null");
        if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_gpu_radiance_rays before rt_gpu_upload_scene");
        if (q->n < 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: negative ray count");
        if (q->mode != RT_MODE_PATH && q->mode != RT_MODE_PREVIEW && q->mode != RT_MODE_WHITTED)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: mode must be RT_MODE_PATH, RT_MODE_PREVIEW or RT_MODE_WHITTED");
        if (q->traverse != RT_TRAVERSE_EXACT && q->traverse != RT_TRAVERSE_CULLED) return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: unknown traverse");
        if (q->max_bounce < 0 || q->max_bounce > RT_MAX_PATH_DEPTH) return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: max_bounce must be in [0, 32]");
        if (q->mode == RT_MODE_PATH && ctx->needs_table && ctx->scene.num_unit_vectors == 0)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: scene has Diffuse materials but no unit-vector table (rt_host_set_unit_vectors)");
        // rounds: one mesh walk per round; a path needs at most (segments) x (mesh shapes) walks (as render_tile counts)
        int mesh_shapes = 0;
        for (int i = 0; i < ctx->scene.num_shapes; i++) mesh_shapes += ctx->host_shape_is_mesh[i] ? 1 : 0;
        const int segments = q->mode == RT_MODE_PATH ? (q->max_bounce > 0 ? q->max_bounce : 1)
                           : q->mode == RT_MODE_WHITTED ? 1 + ctx->scene.num_lights : 1;
        const int rounds = segments * (mesh_shapes > 0 ? mesh_shapes : 1);
        if (rounds >= RT_MAX_ROUNDS) return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: segments x mesh shapes exceed the round table");
        if (q->n == 0) return RT_OK;
        if (!q->rays || !q->rgba) return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: rays and rgba are required");
        RT_CUDA(cudaSetDevice(ctx->device));
        const void* ptrs[3] = { q->rays, q->rng_stream, q->rgba };
        const char* names[3] = { "rays", "rng_stream", "rgba" };
        for (int k = 0; k < 3; k++)
            if (ptrs[k] && !on_device(ctx, ptrs[k]))
                return fail(ctx, RT_ERR_INVALID, std::string("rt_gpu_radiance_rays: ") + names[k] + " is not device memory of the context's GPU");
        // (the samples are written as float4)
        if ((uintptr_t)q->rgba % 16 != 0 || (uintptr_t)q->rays % 4 != 0 || (uintptr_t)q->rng_stream % 4 != 0)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_radiance_rays: rgba must be 16-byte aligned, rays and rng_stream 4-byte aligned");
        int rc = init_walk_grid(ctx);
        if (rc != RT_OK) return rc;
        const size_t n = (size_t)q->n;
        const size_t levels = q->mode == RT_MODE_PATH ? (size_t)(q->max_bounce > 0 ? q->max_bounce : 1) : 1;
        const bool whitted = q->mode == RT_MODE_WHITTED;
        size_t pool_want = 0;
        if ((rc = plan_pools(ctx, (n + 255) & ~(size_t)255, levels, whitted, &pool_want)) != RT_OK) return rc;
        if ((rc = grow_pools(ctx, pool_want, levels, whitted)) != RT_OK) return rc;
        const size_t piece = pool_want & ~(size_t)31;   // path_alloc_packet takes 32 ids per warp with a live ray

        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        const bool cull = q->traverse == RT_TRAVERSE_CULLED;
        RenderArgs a;
        memset(&a, 0, sizeof a);
        a.mode = q->mode;
        a.max_bounce = q->max_bounce;
        a.seed = q->seed;
        a.q_sample = q->sample;
        a.q_first_draw = q->first_draw;
        a.height = 1;
        a.counters = ctx->counters;
        a.exact = cull ? 0 : 1;
        a.all_bounded = ctx->all_bounded ? 1 : 0;
        return enqueue_ray_batch(ctx, a, n, piece, q->mode, rounds, mesh_shapes > 0, cull, st,
                                 [&](RenderArgs& pa, size_t begin, size_t count) {
                                     pa.q_rays = q->rays + 7 * begin;
                                     pa.q_stream = q->rng_stream ? q->rng_stream + begin : nullptr;
                                     pa.q_stream_base = q->rng_stream_base + (uint32_t)begin;
                                     pa.samples = reinterpret_cast<float4*>(q->rgba + 4 * begin);
                                     pa.width = (int)count;
                                 });
    });
}

int rt_gpu_synchronize(rt_gpu_ctx* ctx)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        return RT_OK;
    });
}

int rt_gpu_readback(rt_gpu_ctx* ctx, int what, void* dst, size_t bytes)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!dst) return fail(ctx, RT_ERR_INVALID, "dst is null");
        RT_CUDA(cudaSetDevice(ctx->device));
        const size_t n = (size_t)ctx->width * ctx->height;
        const void* src = nullptr; size_t need = 0;
        switch (what)
        {
        case RT_READ_ACCUM_RGBN_F32: src = ctx->accum; need = n * sizeof(float4); break;
        case RT_READ_DISPLAY_ARGB8: src = ctx->display; need = n * sizeof(uint32_t); break;
        case RT_READ_PRIMARY_IDS_I32X2: src = ctx->prim_ids; need = n * sizeof(int2); break;
        case RT_READ_PRIMARY_DIST_F32: src = ctx->prim_dist; need = n * sizeof(float); break;
        case RT_READ_COUNTERS_U64: src = ctx->counters; need = sizeof(rt_counters); break;
        case RT_READ_PREVIEW_RGBA_F32:
            if (!ctx->preview) return fail(ctx, RT_ERR_NO_SCENE, "no preview pass has been rendered on this frame");
            src = ctx->preview; need = n * sizeof(float4); break;
        default: return fail(ctx, RT_ERR_INVALID, "unknown readback selector");
        }
        if (what != RT_READ_COUNTERS_U64 && n == 0) return fail(ctx, RT_ERR_NO_SCENE, "no frame buffers yet (render or reset_accum first)");
        if (bytes < need) return fail(ctx, RT_ERR_SIZE, "readback buffer too small");
        RT_CUDA(cudaMemcpyAsync(dst, src, need, cudaMemcpyDeviceToHost, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        return RT_OK;
    });
}

int rt_gpu_last_render_ms(rt_gpu_ctx* ctx, float* out_ms)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx || !out_ms) return RT_ERR_INVALID;
        if (!ctx->timed) return fail(ctx, RT_ERR_INVALID, "no render has been enqueued");
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(cudaEventSynchronize(ctx->ev1));
        RT_CUDA(cudaEventElapsedTime(out_ms, ctx->ev0, ctx->ev1));
        return RT_OK;
    });
}

int rt_gpu_last_kernel_ms(rt_gpu_ctx* ctx, float* out_ms, int32_t* out_launches)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx || !out_ms) return RT_ERR_INVALID;
        if (!ctx->timed) return fail(ctx, RT_ERR_INVALID, "no render has been enqueued");
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(cudaEventSynchronize(ctx->ev1));
        float total = 0.0f;
        for (int k = 0; k + 1 < ctx->kev_used; k += 2)
        {
            float ms = 0.0f;
            RT_CUDA(cudaEventElapsedTime(&ms, ctx->kev[k], ctx->kev[k + 1]));
            total += ms;
        }
        *out_ms = total;
        if (out_launches) *out_launches = ctx->kev_used / 2;
        return RT_OK;
    });
}

int rt_gpu_kernel_class_ms(rt_gpu_ctx* ctx, float* ms, int32_t* launches, int32_t num_classes)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx || !ms || !launches || num_classes <= 0) return RT_ERR_INVALID;
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(sync_all_streams(ctx));
        for (int c = 0; c < num_classes; c++) { ms[c] = 0.0f; launches[c] = 0; }
        for (int k = 0; k + 1 < ctx->cev_used; k++)
        {
            const int cls = ctx->cev_cls[k];
            if (cls < 0 || cls >= num_classes) continue;
            float t = 0.0f;
            RT_CUDA(cudaEventElapsedTime(&t, ctx->cev[k], ctx->cev[k + 1]));
            ms[cls] += t; launches[cls]++;
        }
        return RT_OK;
    });
}

int rt_gpu_reset_counters(rt_gpu_ctx* ctx)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        RT_CUDA(cudaSetDevice(ctx->device));
        RT_CUDA(cudaMemsetAsync(ctx->counters, 0, sizeof(rt_counters), ctx->stream));
        return RT_OK;
    });
}

int rt_gpu_resolve_display(rt_gpu_ctx* ctx)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        const int n = ctx->width * ctx->height;
        if (n == 0) return fail(ctx, RT_ERR_NO_SCENE, "no frame buffers yet");
        RT_CUDA(cudaSetDevice(ctx->device));
        rt_display_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->accum, ctx->display, n);
        RT_CUDA(cudaGetLastError());
        ctx->launches++;
        return RT_OK;
    });
}

void* rt_gpu_stream(rt_gpu_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }


void* rt_gpu_accum_device_ptr(rt_gpu_ctx* ctx) { return ctx ? (void*)ctx->accum : nullptr; }

uint64_t rt_gpu_launch_count(rt_gpu_ctx* ctx) { return ctx ? ctx->launches : 0; }

// experiment knobs (tools/, tests that force the long-walk path); the defaults are what ships
static void tuning_from_env(rt_gpu_ctx* ctx)
{
    if (getenv("RT_FINISH_ROUND")) ctx->tune_finish_round = atoi(getenv("RT_FINISH_ROUND"));
    if (getenv("RT_LONG_LIMIT")) ctx->tune_long_limit = (unsigned)atoi(getenv("RT_LONG_LIMIT"));
    if (getenv("RT_SMALL_ROUND")) ctx->tune_small_round = (unsigned)atoi(getenv("RT_SMALL_ROUND"));
    if (getenv("RT_THIN_COUNT")) ctx->tune_thin_count = (unsigned)atoi(getenv("RT_THIN_COUNT"));
    if (getenv("RT_LONG_GROUP_N")) ctx->tune_long_group = atoi(getenv("RT_LONG_GROUP_N"));
    if (getenv("RT_PACKET_ROUNDS")) ctx->tune_packet_rounds = atoi(getenv("RT_PACKET_ROUNDS"));
    if (getenv("RT_PACKET_PROBE")) ctx->tune_packet_probe = (unsigned)atoi(getenv("RT_PACKET_PROBE"));
    if (getenv("RT_PACKET_MIN_LANES")) ctx->tune_packet_min_lanes = (unsigned)atoi(getenv("RT_PACKET_MIN_LANES"));
    if (getenv("RT_THIN_LIMIT")) ctx->tune_thin_limit = (unsigned)atoi(getenv("RT_THIN_LIMIT"));
    if (getenv("RT_SAMPLE_BUDGET_MB")) ctx->tune_sample_budget = (size_t)atoi(getenv("RT_SAMPLE_BUDGET_MB")) << 20;
    ctx->tune_time_long = getenv("RT_TIME_LONG") != nullptr;
    if (getenv("RT_FEW_CHUNKS")) ctx->tune_few_chunks = atoi(getenv("RT_FEW_CHUNKS"));
    if (getenv("RT_TOP_STAGE")) ctx->tune_top_stage = atoi(getenv("RT_TOP_STAGE")) != 0;
    if (getenv("RT_OCTO")) ctx->tune_octo = atoi(getenv("RT_OCTO")) != 0;
    if (getenv("RT_THIN_FROM_ROUND")) ctx->tune_thin_from_round = atoi(getenv("RT_THIN_FROM_ROUND"));   // k > 0: from round k; -1: never
    if (getenv("RT_THIN_GRID_COUNT")) ctx->tune_thin_grid_count = (unsigned)atoi(getenv("RT_THIN_GRID_COUNT"));
}

int rt_gpu_set_tuning(rt_gpu_ctx* ctx, int32_t window_items, int32_t min_lanes, int32_t leaf_wait, int32_t pool_kpaths)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (window_items < 32 || window_items % 32 != 0 || min_lanes < 1 || min_lanes > 32)
            return fail(ctx, RT_ERR_INVALID, "window_items must be a positive multiple of 32, min_lanes in [1, 32]");
        ctx->tune_window = (unsigned)window_items;
        ctx->tune_min_lanes = min_lanes;
        ctx->tune_leaf_wait = leaf_wait < 0 ? 0 : (leaf_wait > 32 ? 32 : leaf_wait);
        if (pool_kpaths > 0) ctx->max_pool_paths = (size_t)pool_kpaths << 10;
        tuning_from_env(ctx);
        return RT_OK;
    });
}

int rt_gpu_time_kernels(rt_gpu_ctx* ctx, int32_t on)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        ctx->time_walks = on == 1;
        ctx->time_classes = on == 2;
        return RT_OK;
    });
}

int rt_gpu_set_pipes(rt_gpu_ctx* ctx, int32_t pipes)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (pipes < 0 || pipes > RT_PIPES) return fail(ctx, RT_ERR_INVALID, "pipes out of range");
        ctx->tune_pipes = pipes == 0 ? RT_PIPES : pipes;      // 0: back to the default
        return RT_OK;
    });
}

int rt_gpu_get_pipes(rt_gpu_ctx* ctx) { return ctx ? ctx->tune_pipes : 0; }

uint64_t rt_gpu_scene_bytes(rt_gpu_ctx* ctx) { return ctx ? (uint64_t)ctx->scene_bytes : 0; }

} // extern "C"
