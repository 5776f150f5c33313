// rt_wave_types.hpp — work-list geometry, the path pool and the per-launch argument blocks of the wavefront
// (shared by the kernels in rt_wave_kernels.cuh and the host side of the boundary in rt_gpu.cu).
#pragma once
#include "rt_device.cuh"

using namespace rtdev;

#define RT_WORK_WINDOW 32u                  // queue entries a warp takes from the round's pop cursor at once
#define RT_POOL_MAX_PATHS (32u << 20)       // path records per pool (~0.5 KB each with a 10-level stack)
#define RT_LEAF_WAIT 18                     // leaves that wait before the walkers are interrupted
#define RT_MIN_LANES 28                     // refill threshold of the mesh walk
#define RT_SAMPLE_BUDGET_BYTES (3ull << 30) // sample buffer cap; longer calls are split in pass chunks
#define RT_SAMPLE_BUDGET_FEW_BYTES (12ull << 30)    // the cap for calls of fewer than RT_FEW_ITEMS camera rays (two chunks)
#define RT_FEW_ITEMS 400000000ull

// ---- work-list geometry ----------------------------------------------------------------------------
struct RenderArgs
{
    int width, height, start, end, mode, max_bounce, antialias;
    uint32_t seed;
    int pass_begin;             // first pass of this chunk
    int spp;                    // samples per pass: 4 (antialias) or 1
    int num_samples;            // pass_count_chunk * spp
    // pixel blocks
    int tiled;                  // 0: one region (rows row0..), 1: round-robin tiles
    int row0, rows;             // untiled region
    int tile_size, tile_count, tile_rank, tiles_x;
    int blocks_x;               // 8-wide blocks per region/tile row
    int blocks_per_tile;
    unsigned num_blocks;
    unsigned num_items;         // num_samples * num_blocks * 32 (the host keeps it below 2^32)
    float4* samples;            // [num_samples][width*height]
    float4* accum;
    float4* preview;            // RT_MODE_PREVIEW: linear colour of the pass (the reference only writes bitcolor then)
    uint32_t* display;
    int2* prim_ids;
    float* prim_dist;
    unsigned long long* counters;
    int exact;                  // traverse == RT_TRAVERSE_EXACT: node_tests/tri_tests are the visits
    int all_bounded;            // every shape has culling bounds (no plane): rays that miss them all see the sky
    // ray queries (rt_gpu_query_rays, modes RT_QMODE_*): the caller's rays and result arrays, indexed by the ray's
    // place in the batch (PathState::pixel); q_tri / q_hit may be null
    const float* q_rays;
    int q_count;
    int* q_shape;
    int* q_tri;
    float* q_hit;
    // radiance queries (rt_gpu_radiance_rays, modes RT_MODE_PATH / PREVIEW / WHITTED): ray i draws from
    // rt_rng_key(seed, stream_i, q_sample) starting at draw q_first_draw, stream_i = q_stream[i] or q_stream_base + i
    const uint32_t* q_stream;
    uint32_t q_stream_base;
    uint32_t q_sample;
    uint32_t q_first_draw;
    // masked renders (rt_gpu_render_masked): the task's work items (block << 5 | lane) whose pixel the mask selects, in
    // block order, and their number (device memory, written by the compaction on the slot's stream)
    const unsigned* list;
    const unsigned* list_count;
    float4* moments;            // rt_gpu_track_moments: {M2.rgb, passes} per pixel, updated by the folds of the *_moments variants
    float4* guide;              // RT_MODE_GUIDES: {HitNormal.xyz, 0} of the nearest hit per pixel (zeros on a miss)
};

// Internal modes of the wavefront kernels next to the RT_MODE_* of the ABI: a batch of ray queries.  A completed
// query writes its result and ends (no shading); ANY is the shadow query (pool record bit 256).  Values the ABI's modes
// do not use.
#define RT_QMODE_NEAREST 8
#define RT_QMODE_ANY 9

// The modes that trace one un-jittered camera ray per pixel and write the primary hit (no samples, no fold)
#define RT_PRIMARY_LIKE(m) ((m) == RT_MODE_PRIMARY || (m) == RT_MODE_GUIDES)

__device__ __forceinline__ bool owns_pixel(const RenderArgs& a, int x, int y)
{
    if (!a.tiled) return true;
    int tile = (y / a.tile_size) * a.tiles_x + x / a.tile_size;
    return tile % a.tile_count == a.tile_rank;
}

// block index + lane -> pixel (or -1 when the lane falls outside the region / image / task range)
__device__ __forceinline__ int block_pixel(const RenderArgs& a, unsigned block, int lane, int& x, int& y)
{
    x = 0; y = 0;
    int ox, oy, w, h, b;
    if (a.tiled)
    {
        unsigned k = block / (unsigned)a.blocks_per_tile;
        b = (int)(block - k * (unsigned)a.blocks_per_tile);
        int tile = a.tile_rank + (int)k * a.tile_count;
        ox = (tile % a.tiles_x) * a.tile_size; oy = (tile / a.tiles_x) * a.tile_size;
        w = a.tile_size; h = a.tile_size;
    }
    else { b = (int)block; ox = 0; oy = a.row0; w = a.width; h = a.rows; }
    int bx = b % a.blocks_x, by = b / a.blocks_x;
    int lx = bx * 8 + (lane & 7), ly = by * 4 + (lane >> 3);
    if (lx >= w || ly >= h) return -1;
    x = ox + lx; y = oy + ly;
    if (x >= a.width || y >= a.height) return -1;
    int pixel = y * a.width + x;
    if (pixel < a.start || pixel > a.end) return -1;
    return pixel;
}

__device__ __forceinline__ void flush_counters(const Counters& c, unsigned long long* g, int exact)
{
    unsigned long long v[7] = { c.rays, c.camera_rays, c.shadow_rays, c.node_visits, c.tri_visits, c.mesh_hits, c.mesh_walks };
#pragma unroll
    for (int k = 0; k < 7; k++)
    {
        unsigned long long x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(RT_FULL_MASK, x, o);
        v[k] = x;
    }
    if ((threadIdx.x & 31) == 0)
    {
        // rt_counters: rays, camera_rays, shadow_rays, node_tests, tri_tests, node_visits, tri_visits, mesh_hits, mesh_walks
        if (v[0]) atomicAdd(g + 0, v[0]);
        if (v[1]) atomicAdd(g + 1, v[1]);
        if (v[2]) atomicAdd(g + 2, v[2]);
        if (v[3]) { atomicAdd(g + 5, v[3]); if (exact) atomicAdd(g + 3, v[3]); }
        if (v[4]) { atomicAdd(g + 6, v[4]); if (exact) atomicAdd(g + 4, v[4]); }
        if (v[5]) atomicAdd(g + 7, v[5]);
        if (v[6]) atomicAdd(g + 8, v[6]);
    }
}

// ---- path pool ---------------------------------------------------------------------------------------
// Every camera ray that cannot be retired on the spot becomes a PATH with a record in this pool
// (structure of arrays, one 16-byte word per field group so a warp reads/writes whole lines).
// Queues hold path ids; a path keeps its id for its whole life.
struct PathPool
{
    float4* ro;         // TestRay origin, .w = current Distance (shrinks as hits are accepted)
    float4* rd;         // direction, .w = Distance of the segment as it was shot
    int4* cur;          // x: shape cursor si, y: best leaf slot, z: state | any << 8 | sky_on_miss << 9, w: hit shape
    float4* bp;         // position of the last accepted triangle
    float4* h0;         // RayHitResult: HitPosition, Distance
    float4* h1;         //               HitNormal, SampledAlpha
    float4* h2;         //               SampledColor, .w = triangle id of the hit (int bits)
    int4* pa;           // pixel, sample slot, rng key, rng draw counter
    int4* pb;           // depth_left, stack height, pass-through mask, light cursor
    float4* w0;         // Whitted only: primary hit position / normal / surface colour / running sum
    float4* w1;
    float4* w2;
    float4* w3;
    float4* st0;        // unwinding stack, [level * cap + path]: att.xyz col.x | col.yz emi.xy | emi.z
    float4* st1;
    float* st2;
    unsigned cap;
};

struct PathState
{
    int pixel, slot;
    Rng rng;
    int depth_left, sp;
    unsigned pass_mask;
    int light;
    float seg_dist;
    float3 w_pos, w_nrm, w_surface, w_sum;
};

struct WaveArgs
{
    PathPool pool;
    unsigned* queue[2];         // path ids of round r live in queue[r & 1]
    unsigned* counts;           // counts[r]: entries of round r;  counts[RT_MAX_ROUNDS]: paths allocated
    unsigned* heads;            // heads[r]: pop cursor of the walk kernel in round r
    unsigned* longq;            // walks the walk kernel gave up on (too long): finished one-warp-per-walk
    unsigned* lcounts;          // lcounts[r] / lheads[r]: entries and pop cursor of longq in round r
    unsigned* lheads;
    unsigned long_limit;        // node steps after which a lane hands its walk to the long-walk kernel
    unsigned thin_count;        // a round with fewer entries than this is latency-bound (its longest walk decides):
    unsigned thin_limit;        //   its walks are parked after thin_limit steps already
    unsigned* slowq;            // walks the packet kernel hands back to the lane-per-walk kernel (incoherent packets)
    unsigned* scounts;          // scounts[r], sheads[r]: that queue's size and pop cursor in round r
    unsigned* sheads;
    unsigned packet_probe;      // a packet is judged every this many steps:
    unsigned packet_min_lanes;  //   fewer lane-tests than packet_min_lanes (of 32, scaled to the packet's rays) per step -> not coherent
    int packets;                // round 0 is allocated in aligned packets of 32 (one generate warp each)
    unsigned small_round;       // a round with fewer entries than this is walked entirely one-warp-per-walk
    unsigned item_begin, item_count;   // slice of the work list this batch generates
    const unsigned* retry_in;          // retry pass: the items to generate (else null) and how many
    const unsigned* retry_in_count;
    unsigned* retry_out;               // items that found the pool full
    unsigned* retry_out_count;
    int min_lanes, leaf_wait;
    unsigned window;
};

#define RT_MAX_ROUNDS 512
#ifndef RT_PIPES
#define RT_PIPES 4
#endif
#define RT_MAX_RETRIES 64
#define RT_SEEN_ROUNDS 64                     // round sizes remembered per pipe (grid sizing of late rounds)
#define RT_SMALL_RETRY 100000u              // a retry pass that had fewer items than this last time is launched with one CTA per SM
#define RT_THIN_GRID_COUNT 600000u           // a round that held fewer entries last time is launched with quarter grids (frames in flight)
#define RT_FRAME_SLOTS 4                     // frames in flight (rt_gpu_set_frame_slot)
#define RT_SMALL_ROUND 24000u               // rounds thinner than this are walked one-warp-per-walk only (frontier kernel)
#ifndef RT_SHADE_BLOCKS
#define RT_SHADE_BLOCKS 2
#endif
#ifndef RT_GEN_BLOCKS
#define RT_GEN_BLOCKS 3
#endif
#define RT_LONG_LIMIT 2048u                 // node steps after which a lane parks its walk for the long-walk kernel
#define RT_THIN_COUNT 200000u               // rounds thinner than this park after RT_THIN_LIMIT steps (0 = never):
#define RT_PACKET_PROBE 24u                 // a packet is judged every this many steps ...
#define RT_PACKET_MIN_LANES 10u             // ... and goes on lane by lane if fewer lanes than this tested a node per step
#define RT_THIN_LIMIT 256u                  //   their time is their longest walk, and the frontier kernel shortens exactly that
#ifndef RT_LONG_BLOCKS
#define RT_LONG_BLOCKS 4
#endif
#ifndef RT_LEAF_SLOTS
#define RT_LEAF_SLOTS 2                     // leaves a lane may hold before its walk has to wait for the triangle phase
#endif
#ifndef RT_STEPS_PER_VOTE
#define RT_STEPS_PER_VOTE 3                  // node steps of the lane-per-walk kernel between two warp votes
#endif
#ifndef RT_WALK_BLOCKS
#define RT_WALK_BLOCKS 4                    // resident 256-thread CTAs per SM of the walk kernel (64 registers)
#endif
#ifndef RT_LONG_GROUP
#define RT_LONG_GROUP 32
#endif
#define RT_FW_INTS_PER_LANE 16              // stack and leaf list hold 16 x G entries each (32 KB per block together)
