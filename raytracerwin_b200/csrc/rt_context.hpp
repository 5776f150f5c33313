// rt_context.hpp — the opaque context behind include/rt_gpu.h and the error and argument helpers every translation
// unit of the library uses (rt_gpu.cu: lifetime / upload / render / queries / readback; rt_scene_edit.cu: scene edits;
// rt_adaptive.cu: moments, mask compaction and pixel selection; rt_denoise.cu: the guided denoiser; rt_exchange.cu: multi-GPU tile exchange; rt_hooks.cu: test and tooling hooks; rt_bvh_build.cu: device BVH builder).
#pragma once
#include "rt_wave_types.hpp"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <initializer_list>
#include <new>
#include <string>
#include <vector>

// Adaptive sampling state of one frame slot (rt_gpu_track_moments, rt_gpu_render_masked, rt_gpu_select_pixels)
struct SlotAdaptive
{
    float4* moments = nullptr;                  // width*height {M2.r, M2.g, M2.b, passes}; allocated by the first track_moments(on)
    bool track = false;                         // the folds of PATH / WHITTED renders update `moments`
    // scratch of a masked render: the device count, the compacted work items of the mask and CUB's temporaries (only grows,
    // stream-ordered on the slot's stream)
    void* scratch = nullptr;
    size_t scratch_cap = 0;
};

// Denoising state of one frame slot (RT_MODE_GUIDES, rt_gpu_denoise)
struct SlotDenoise
{
    float4* guide = nullptr;                    // width*height {HitNormal.xyz, 0} of the nearest hit (allocated by the first GUIDES call)
    bool guides = false;                        // a GUIDES render has been enqueued since the frame was (re)allocated
    // the filter's per-pixel records and ping-pong buffers (only grows, stream-ordered on the slot's stream)
    void* scratch = nullptr;
    size_t scratch_cap = 0;
};

struct rt_gpu_ctx
{
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    // per-launch timing of the path kernel inside the last render_tile (one pair per pass chunk)
    std::vector<cudaEvent_t> kev;
    int kev_used = 0;
    std::string err;
    int num_sms = 0;

    bool has_scene = false;
    bool needs_table = false;                   // scene has Diffuse materials (RandomHemisphereDirection)
    DevScene scene;
    std::vector<void*> scene_allocs;
    std::vector<cudaArray_t> arrays;
    std::vector<cudaTextureObject_t> texobjs;
    std::vector<DevTexture> host_textures;      // flat list of every texture (test hook)
    std::vector<char> host_shape_is_mesh;
    bool all_bounded = false;
    size_t scene_bytes = 0;
    size_t texel_upload_bytes = 0;              // host-to-device bytes the last upload spent on texels

    int width = 0, height = 0;
    float4* accum = nullptr;
    uint32_t* display = nullptr;
    int2* prim_ids = nullptr;
    float* prim_dist = nullptr;
    float4* preview = nullptr;                  // linear colour of the last preview pass (allocated by the first RT_MODE_PREVIEW call)
    SlotAdaptive adapt;
    SlotDenoise den;
    unsigned long long* counters = nullptr;     // rt_counters
    // Frame slots (rt_gpu_set_frame_slot): the members above — stream, timing events, frame size, the five frame
    // buffers, the adaptive and the denoising state — are those of the CURRENT slot; the other slots' sets wait here.  Calls that
    // address different slots are not ordered against each other on the device, so a driver can enqueue frame k+1
    // while the thin last bounce rounds, the exchange and the read-back of frame k are still running.
    struct FrameSlot
    {
        cudaStream_t stream = nullptr;
        cudaEvent_t ev0 = nullptr, ev1 = nullptr;
        bool timed = false;
        int width = 0, height = 0;
        float4* accum = nullptr; uint32_t* display = nullptr; int2* prim_ids = nullptr; float* prim_dist = nullptr; float4* preview = nullptr;
        SlotAdaptive adapt;
        SlotDenoise den;
    };
    FrameSlot parked[RT_FRAME_SLOTS];
    int slot = 0;
    unsigned slot_mask = 1u; int slots_touched = 1;   // which slots a driver has addressed so far
    bool slots_used = false;                    // rt_gpu_set_frame_slot has been called: calls rotate through the pipes
    int pipe_cursor = 0;
    // wavefront state: path pool, round queues, round counters
    // Batches of a call are dealt round-robin to RT_PIPES pipes, each with its own stream, pool and
    // queues, so the thin late rounds of one batch (few long walks: latency bound) overlap the
    // dense early rounds of the next.
    struct Pipe
    {
        cudaStream_t stream = nullptr;
        cudaEvent_t done = nullptr;
        PathPool pool;
        unsigned* queue[2] = { nullptr, nullptr };
        unsigned* round_counters = nullptr;     // counts[RT_MAX_ROUNDS + 1] then heads[RT_MAX_ROUNDS]
        unsigned* longq = nullptr;              // parked long walks of the current round
        unsigned* slowq = nullptr;              // walks of incoherent packets, handed to the lane-per-walk kernel
        unsigned* retry[2] = { nullptr, nullptr };   // items turned away by a full pool (ping-pong)
        unsigned* retry_counts = nullptr;       // one per retry pass
        unsigned* seen_counts = nullptr;        // PINNED HOST copy of the round sizes of the last batch on this pipe (first generate pass)
        unsigned long long seen_signature = 0;  // which call shape they belong to
        volatile unsigned* seen_retry = nullptr;   // PINNED HOST copy of the retry-list sizes of that batch (items each generate pass turned away)
        float4* samples = nullptr;              // radiance samples of the chunk this pipe is rendering
        size_t samples_cap = 0;                 // float4s
        size_t retry_cap = 0;
        std::vector<void*> allocs;
    };
    Pipe pipes[RT_PIPES];
    cudaEvent_t fork = nullptr;
    size_t pool_cap = 0, pool_levels = 0;       // per pipe
    bool pool_whitted = false;
    size_t max_pool_paths = RT_POOL_MAX_PATHS;  // per call, over all pipes
    int tune_pipes = RT_PIPES;
    int walk_blocks_per_sm = 0;
    struct TileTable { int width, height, tile_size, tile_count, rank; long long* offsets; };
    std::vector<TileTable> tile_tables;
    float4* gather_staging = nullptr;
    size_t gather_staging_cap = 0;
    unsigned long long launches = 0;            // kernels launched by this context
    unsigned tune_window = RT_WORK_WINDOW;
    int tune_min_lanes = RT_MIN_LANES;
    int tune_leaf_wait = RT_LEAF_WAIT;
    bool time_walks = false;                    // record an event pair around every walk launch (rt_gpu_time_kernels)
    bool time_classes = false;                  // rt_gpu_time_kernels(ctx, 2): one event before every launch, by kernel class
    std::vector<cudaEvent_t> cev;
    std::vector<int> cev_cls;
    int cev_used = 0;
    unsigned tune_long_limit = RT_LONG_LIMIT;
    unsigned tune_small_round = RT_SMALL_ROUND;
    unsigned tune_thin_count = RT_THIN_COUNT;
    int tune_long_group = RT_LONG_GROUP;
    int tune_packet_rounds = -1;            // -1: by mode
    unsigned tune_packet_probe = RT_PACKET_PROBE;
    unsigned tune_packet_min_lanes = RT_PACKET_MIN_LANES;
    unsigned tune_thin_limit = RT_THIN_LIMIT;
    int tune_thin_from_round = 0;               // RT_THIN_FROM_ROUND: 0 = by the sizes last seen (frames in flight only), k > 0 = from round k, -1 = never
    unsigned tune_thin_grid_count = RT_THIN_GRID_COUNT;   // a round that had fewer entries than this gets quarter grids
    int tune_few_chunks = 0;                    // RT_FEW_CHUNKS: pass chunks of a call of few camera rays (0: 2, or 1 with frame slots)
    size_t tune_sample_budget = 0;              // RT_SAMPLE_BUDGET_MB at create (0: by call size)
    bool tune_time_long = false;                // RT_TIME_LONG at create: timed brackets span walk + long walk

    // ---- scene updates (rt_gpu_update_mesh / rt_gpu_refit_mesh / rt_gpu_replace_mesh / rt_gpu_update_shapes) ----
    // What the updates check and swap, per uploaded shape and mesh.  A mesh's arrays are double-buffered from its first
    // update on: an update builds into the spare set and publishes it; the published set becomes the spare.
    std::vector<rt_shape> host_shapes;          // the records as uploaded (materials follow rt_gpu_update_shapes)
    // ---- appearance updates (rt_gpu_update_materials / rt_gpu_update_lights / rt_gpu_update_texture) ----
    std::vector<rt_material> host_materials;    // the graph the device holds (the checks of an update run on its edit)
    // Room of ctx->scene.materials / .lights in records.  `pooled`: from cudaMallocAsync by an update, released with
    // cudaFreeAsync when a larger array replaces it; the uploaded arrays (cudaMalloc) stay until the next upload or destroy.
    int material_cap = 0, light_cap = 0;
    bool materials_pooled = false, lights_pooled = false;
    std::vector<std::vector<DevTexture>> mesh_textures;   // per mesh, per slot: the atlas rectangle (0 x 0: no pixels)
    cudaArray_t atlas_array = nullptr;          // in `arrays`
    cudaSurfaceObject_t atlas_surface = 0;      // writes into the atlas (8-bit expansion); destroyed with the scene
    // One set of a mesh's arrays: room for `cap` triangles (2 * cap - 1 nodes).  `pooled`: from cudaMallocAsync by an
    // update, released with cudaFreeAsync when a larger set replaces it; the uploaded set (cudaMalloc) stays in
    // scene_allocs until the next upload or destroy.
    struct MeshArrays { rt_bvh_node* nodes; rt_tri* tris; rt_shade* shade; int cap; bool pooled; };
    struct MeshState
    {
        int num_tris = 0;                       // published counts: as uploaded, then those of the last replace
        int num_nodes = 0;                      // as uploaded: an update builds 2 * num_tris - 1
        int users = 0;                          // shapes that reference the mesh
        // The published tree is a full binary tree over all its nodes whose leaves name every triangle slot exactly once
        // (checked at upload, true after an update): what rt_gpu_refit_mesh needs to reach and rewrite every node.
        bool refittable = false;
        MeshArrays cur = { nullptr, nullptr, nullptr, 0, false };      // published (shade in leaf order)
        MeshArrays spare = { nullptr, nullptr, nullptr, 0, false };    // allocated by the first update
    };
    std::vector<MeshState> mesh_state;
    // Recorded by every update after it has published; every later scene reader waits for it on its stream.  Live from
    // the first update of an upload on (no update: no event, no wait).
    cudaEvent_t scene_event = nullptr;
    bool scene_event_live = false;
    cudaEvent_t join_event = nullptr;           // one record per context stream when an update publishes
    void* update_scratch = nullptr;             // the builder's scratch block and the update's temporaries (only grows)
    size_t update_scratch_cap = 0;
    int* update_counts = nullptr;               // PINNED HOST: the builder's per-level read
    cudaEvent_t order_event = nullptr;          // orders a caller's stream and the slot's stream (render_masked, select_pixels, denoise)
};

// A scene reader enqueued on `st` runs after the last published update
static inline cudaError_t wait_scene(const rt_gpu_ctx* ctx, cudaStream_t st)
{
    return ctx->scene_event_live ? cudaStreamWaitEvent(st, ctx->scene_event, 0) : cudaSuccess;
}

extern thread_local std::string g_create_error;

static inline int fail(rt_gpu_ctx* c, int code, const std::string& msg)
{
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

#define RT_CUDA(call)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return fail(ctx, RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
    } while (0)

// No C++ exception crosses the C ABI (include/rt_gpu.h: every entry returns 0 or a negative rt_status): the
// bodies of the entry points that allocate host memory (std::vector / std::string) run inside this guard.
template <typename F>
static inline int rt_guard(rt_gpu_ctx* ctx, F&& body) noexcept
{
    try { return body(); }
    catch (const std::bad_alloc&) { try { return fail(ctx, RT_ERR_NOMEM, "out of host memory"); } catch (...) { return RT_ERR_NOMEM; } }
    catch (const std::exception& e) { try { return fail(ctx, RT_ERR_INVALID, e.what()); } catch (...) { return RT_ERR_INVALID; } }
    catch (...) { return RT_ERR_INVALID; }
}

// The caller's arrays of a call that takes device memory (`fn` names the call in the messages): each one given (null:
// an optional array left out) must be `align`-byte aligned device memory (or managed memory) of the context's GPU.
struct DeviceArg { const void* ptr; const char* name; size_t align; };
static inline int check_device_args(rt_gpu_ctx* ctx, const char* fn, std::initializer_list<DeviceArg> args)
{
    for (const DeviceArg& a : args)
    {
        if (!a.ptr) continue;
        if ((uintptr_t)a.ptr % a.align != 0)
            return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": " + a.name + " must be " + std::to_string(a.align) + "-byte aligned");
        cudaPointerAttributes at;
        memset(&at, 0, sizeof at);
        const cudaError_t e = cudaPointerGetAttributes(&at, a.ptr);
        if (e != cudaSuccess) cudaGetLastError();
        if (e != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != ctx->device)
            return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": " + a.name + " is not device memory of the context's GPU");
    }
    return RT_OK;
}

// The material checks of rt_gpu_upload_scene and rt_gpu_update_materials (rt_gpu.cu; library-internal: not exported)
__attribute__((visibility("hidden"))) int check_materials(rt_gpu_ctx* ctx, const rt_material* mats, int n, const std::string& prefix,
                                                          bool* needs_table);

// Work enqueued on `to` after this runs after everything enqueued on `from` before it (no-op when they are one stream)
static inline cudaError_t order_streams(rt_gpu_ctx* ctx, cudaStream_t from, cudaStream_t to)
{
    if (from == to) return cudaSuccess;
    if (!ctx->order_event)
    {
        const cudaError_t e = cudaEventCreateWithFlags(&ctx->order_event, cudaEventDisableTiming);
        if (e != cudaSuccess) return e;
    }
    const cudaError_t e = cudaEventRecord(ctx->order_event, from);
    return e != cudaSuccess ? e : cudaStreamWaitEvent(to, ctx->order_event, 0);
}

// The work items of the task `a` (block << 5 | lane, in block order) whose pixel has mask[pixel] != 0, compacted into the
// slot's scratch on the slot's stream: *list and *count are device addresses (rt_adaptive.cu; library-internal)
__attribute__((visibility("hidden"))) int compact_mask(rt_gpu_ctx* ctx, const RenderArgs& a, const uint8_t* mask,
                                                       const unsigned** list, const unsigned** count);
