// rt_wave_kernels.cuh — the kernels of the wavefront (generate / walk / packet walk / long walk / shade /
// fold).  Included by rt_gpu.cu only (it holds non-template __global__ functions).
// Compiled with -fmad=false; see rt_device.cuh.
#pragma once
#include "rt_wave_types.hpp"

template <int MODE>
__device__ __forceinline__ void pool_store(const PathPool& p, unsigned id, const Query& q, int state, const PathState& s, bool sky_on_miss = false)
{
    p.ro[id] = make_float4(q.r.o.x, q.r.o.y, q.r.o.z, q.r.dist);
    p.rd[id] = make_float4(q.r.d.x, q.r.d.y, q.r.d.z, s.seg_dist);
    p.cur[id] = make_int4(q.si, q.best, state | (q.any ? 256 : 0) | (sky_on_miss ? 512 : 0), q.hit_shape);
    // A query that has hit nothing yet (hit shape -1) still holds the hit record query_begin gave it, and the leaf
    // position is written by the walk kernels: neither is stored (pool_load re-creates them) — 64 of a record's
    // 144 bytes that the common case (a mesh walk straight after the segment began) never moves.
    if (q.hit_shape != -1)
    {
        p.h0[id] = make_float4(q.h.pos.x, q.h.pos.y, q.h.pos.z, q.h.dist);
        p.h1[id] = make_float4(q.h.nrm.x, q.h.nrm.y, q.h.nrm.z, q.h.alpha);
        p.h2[id] = make_float4(q.h.color.x, q.h.color.y, q.h.color.z, __int_as_float(q.tri));
    }
    p.pa[id] = make_int4(s.pixel, s.slot, (int)s.rng.key, (int)s.rng.n);
    p.pb[id] = make_int4(s.depth_left, s.sp, (int)s.pass_mask, s.light);
    if (MODE == RT_MODE_WHITTED)
    {
        p.w0[id] = make_float4(s.w_pos.x, s.w_pos.y, s.w_pos.z, 0.0f);
        p.w1[id] = make_float4(s.w_nrm.x, s.w_nrm.y, s.w_nrm.z, 0.0f);
        p.w2[id] = make_float4(s.w_surface.x, s.w_surface.y, s.w_surface.z, 0.0f);
        p.w3[id] = make_float4(s.w_sum.x, s.w_sum.y, s.w_sum.z, 0.0f);
    }
}

template <int MODE>
__device__ __forceinline__ void pool_load(const PathPool& p, unsigned id, Query& q, int& state, PathState& s)
{
    const float4 ro = p.ro[id], rd = p.rd[id];
    const int4 cur = p.cur[id], pa = p.pa[id], pb = p.pb[id];
    // (see pool_store) hit record: query_begin's unless something was hit; leaf position: only after a walk that found one
    float4 bp = make_float4(0.0f, 0.0f, 0.0f, 0.0f), h0 = bp, h1 = make_float4(0.0f, 0.0f, 0.0f, 1.0f), h2 = make_float4(1.0f, 1.0f, 1.0f, __int_as_float(-1));
    if (cur.w != -1) { h0 = p.h0[id]; h1 = p.h1[id]; h2 = p.h2[id]; }
    if (cur.y >= 0) bp = p.bp[id];
    q.r.o = xyz(ro); q.r.dist = ro.w; q.r.d = xyz(rd); s.seg_dist = rd.w;
    q.pre = ray_pre(q.r);
    q.weird = !(q.pre.ex && q.pre.ey && q.pre.ez && finite3(q.r.o) && finite3(q.r.d));
    q.si = cur.x; q.best = cur.y; state = cur.z & 255; q.any = (cur.z & 256) != 0; q.hit_shape = cur.w;
    q.node = 0;
    q.bpos = xyz(bp); q.tri = __float_as_int(h2.w);
    q.h.pos = xyz(h0); q.h.dist = h0.w; q.h.nrm = xyz(h1); q.h.alpha = h1.w; q.h.color = xyz(h2);
    s.pixel = pa.x; s.slot = pa.y; s.rng.key = (uint32_t)pa.z; s.rng.n = (uint32_t)pa.w;
    s.depth_left = pb.x; s.sp = pb.y; s.pass_mask = (unsigned)pb.z; s.light = pb.w;
    if (MODE == RT_MODE_WHITTED)
    {
        s.w_pos = xyz(p.w0[id]); s.w_nrm = xyz(p.w1[id]); s.w_surface = xyz(p.w2[id]); s.w_sum = xyz(p.w3[id]);
    }
    else { s.w_pos = s.w_nrm = s.w_surface = s.w_sum = V3(0, 0, 0); }
}

// append the calling lanes' path ids to a queue: one atomic per warp (ballot -> leader add -> shuffle)
__device__ __forceinline__ void queue_push(unsigned* queue, unsigned* count, bool push, unsigned id)
{
    const unsigned active = __activemask();
    const unsigned mask = __ballot_sync(active, push);
    if (mask == 0) return;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    unsigned base = 0;
    if (lane == leader) base = atomicAdd(count, (unsigned)__popc(mask));
    base = __shfl_sync(active, base, leader);
    if (push) queue[base + (unsigned)__popc(mask & ((1u << lane) - 1u))] = id;
}

// allocate path ids the same way
__device__ __forceinline__ unsigned path_alloc(unsigned* counter, bool want)
{
    const unsigned active = __activemask();
    const unsigned mask = __ballot_sync(active, want);
    if (mask == 0) return 0;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    unsigned base = 0;
    if (lane == leader) base = atomicAdd(counter, (unsigned)__popc(mask));
    base = __shfl_sync(active, base, leader);
    return base + (unsigned)__popc(mask & ((1u << lane) - 1u));
}

// The same, in whole packets: a warp with at least one taker allocates 32 ids, takers first, so that every
// aligned group of 32 queue entries comes from ONE warp of the generate kernel (one 8x4-pixel block) and
// the packet walk finds coherent rays.  `spare` is the id a non-taker has to mark as unused (or ~0u).
__device__ __forceinline__ unsigned path_alloc_packet(unsigned* counter, bool want, unsigned& spare)
{
    spare = 0xffffffffu;
    const unsigned active = __activemask();
    const unsigned mask = __ballot_sync(active, want);
    if (mask == 0) return 0;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    unsigned base = 0;
    if (lane == leader) base = atomicAdd(counter, 32u);
    base = __shfl_sync(active, base, leader);
    const unsigned below = (1u << lane) - 1u;
    if (!want) spare = base + (unsigned)__popc(mask) + (unsigned)__popc(~mask & below);
    return base + (unsigned)__popc(mask & below);
}

// ---- shading of one completed query ---------------------------------------------------------------------
// RayTracerScene::RayTrace's body after FindIntersectionWithScene (RayTracerScene.cpp:44-97), the
// light loop of the Whitted configuration (CalculateLightColor, :127-175), or the id dump.
// Per-path unwinding record: RayTrace combines the radiance of the NEXT segment as
//   final = 0 + (att * L_next) * SampledColor; final += emissive
// on the way back up its recursion.  The path runs the recursion forwards and keeps (att, colour,
// emissive) per level in the pool so the fold runs in exactly the reference's order and rounding;
// pass-through levels (:79-85, final = 0 + L_next) only set a bit.
// A completed ray query (RT_QMODE_*): its result at the ray's place in the batch, with the fields and the
// zeros-on-a-miss of rt_trace_rays_kernel (rt_hooks.cu).
template <int MODE>
__device__ __forceinline__ void query_result(const RenderArgs& a, int i, const Query& q)
{
    const int shape = q.hit_shape;
    if (MODE == RT_QMODE_ANY) { a.q_shape[i] = shape >= 0 ? 1 : 0; return; }
    a.q_shape[i] = shape;
    if (a.q_tri) a.q_tri[i] = shape >= 0 ? q.tri : -1;
    if (a.q_hit)
    {
        float* o = a.q_hit + 11 * (size_t)i;
        if (shape >= 0)
        {
            o[0] = q.h.pos.x; o[1] = q.h.pos.y; o[2] = q.h.pos.z; o[3] = q.h.nrm.x; o[4] = q.h.nrm.y; o[5] = q.h.nrm.z;
            o[6] = q.h.dist; o[7] = q.h.color.x; o[8] = q.h.color.y; o[9] = q.h.color.z; o[10] = q.h.alpha;
        }
        else
            for (int k = 0; k < 11; k++) o[k] = 0.0f;
    }
}

// Returns true when the path continues with `next` (query not yet begun); otherwise the path has
// ended and its sample has been written.
template <int MODE>
__device__ __forceinline__ bool shade_query(const DevScene& sc, const RenderArgs& a, const PathPool& pool, unsigned id,
                                            const Query& q, PathState& s, Ray& next, bool& next_any)
{
    if (MODE == RT_QMODE_NEAREST || MODE == RT_QMODE_ANY)
    {
        query_result<MODE>(a, s.pixel, q);
        return false;
    }
    bool done = false, newseg = false;
    next_any = false;
    float3 L = V3(0, 0, 0);
    const int shape = q.hit_shape;
    Ray in; in.o = q.r.o; in.d = q.r.d; in.dist = s.seg_dist;
    if (RT_PRIMARY_LIKE(MODE))
    {
        a.prim_ids[s.pixel] = make_int2(shape, shape >= 0 ? q.tri : -1);
        a.prim_dist[s.pixel] = shape >= 0 ? q.h.dist : 0.0f;
        if (MODE == RT_MODE_GUIDES)
            a.guide[s.pixel] = shape >= 0 ? make_float4(q.h.nrm.x, q.h.nrm.y, q.h.nrm.z, 0.0f) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        return false;
    }
    else if (MODE == RT_MODE_WHITTED)
    {
        bool next_light = false;
        if (!q.any)
        {
            if (shape == -1) { L = sky_color(in.d); done = true; }
            else
            {
                s.w_pos = q.h.pos; s.w_nrm = q.h.nrm; s.w_surface = q.h.color; s.w_sum = V3(0, 0, 0);
                s.light = 0; next_light = true;
            }
        }
        else
        {
            // CalculateLightColor: black if occluded, else SurfaceColor * max(0, N.L)
            float3 c = V3(0, 0, 0);
            if (shape == -1) c = mulf3(s.w_surface, max_ref(0.0f, dot3(s.w_nrm, in.d)));
            s.w_sum = add3(s.w_sum, c);
            s.light++; next_light = true;
        }
        if (next_light)
        {
            if (s.light >= sc.num_lights) { L = s.w_sum; done = true; }
            else
            {
                const rt_light* l = sc.lights + s.light;
                float3 ldir = ld3(l->pos_or_dir);
                float dist = 0.0f;
                if (l->type == RT_LIGHT_POINT)
                {
                    ldir = normalized3(sub3(ld3(l->pos_or_dir), s.w_pos));
                    dist = magnitude3(sub3(s.w_pos, ld3(l->pos_or_dir)));
                }
                else if (l->type == RT_LIGHT_DIRECTIONAL) dist = 1000.0f;
                next.o = add3(s.w_pos, mulf3(ldir, sc.bounce_offset)); next.d = ldir; next.dist = dist;
                newseg = true; next_any = true;
            }
        }
    }
    else if (shape == -1) { L = sky_color(in.d); done = true; }
    else
    {
        const int mat = sc.shapes[shape].material;
        if (MODE == RT_MODE_PREVIEW)
        {
            if (mat >= 0)
            {
                Ray unused = in;
                const Bounce b = material_bounce(sc, mat, true, in, q.h, unused, s.rng);
                L = add3(L, mul3(b.att, q.h.color));
            }
            done = true;
        }
        else if (mat < 0) done = true;
        else
        {
            const Bounce b = material_bounce(sc, mat, false, in, q.h, next, s.rng);
            if (rng_random(s.rng) <= q.h.alpha)
            {
                if (is_non_zero(b.att))
                {
                    const size_t k = (size_t)s.sp * pool.cap + id;
                    pool.st0[k] = make_float4(b.att.x, b.att.y, b.att.z, q.h.color.x);
                    pool.st1[k] = make_float4(q.h.color.y, q.h.color.z, b.emi.x, b.emi.y);
                    pool.st2[k] = b.emi.z;
                    s.sp++;
                    newseg = true;
                }
                else { L = add3(L, b.emi); done = true; }
            }
            else
            {
                // alpha pass-through (RayTracerScene.cpp:79-85): same direction, unattenuated
                next.o = add3(q.h.pos, mulf3(in.d, sc.bounce_offset)); next.d = in.d; next.dist = in.dist - q.h.dist;
                s.pass_mask |= 1u << s.sp;
                s.sp++;
                newseg = true;
            }
            if (newseg)
            {
                s.depth_left--;
                // RayTrace(ray, 0) returns black before any query (RayTracerScene.cpp:39-42)
                if (s.depth_left == 0) { newseg = false; done = true; }
            }
        }
    }
    if (done)
    {
        // fold the levels back in recursion order, emit the sample
        for (int k = s.sp - 1; k >= 0; k--)
        {
            if ((s.pass_mask >> k) & 1u) L = add3(V3(0, 0, 0), L);
            else
            {
                const size_t e = (size_t)k * pool.cap + id;
                const float4 s0 = pool.st0[e], s1 = pool.st1[e];
                const float s2 = pool.st2[e];
                const float3 att = V3(s0.x, s0.y, s0.z), col = V3(s0.w, s1.x, s1.y), emi = V3(s1.z, s1.w, s2);
                const float3 f = add3(V3(0, 0, 0), mul3(mul3(att, L), col));
                L = add3(f, emi);
            }
        }
        a.samples[(size_t)s.slot * ((size_t)a.width * a.height) + s.pixel] = make_float4(L.x, L.y, L.z, 0.0f);
        return false;
    }
    return newseg;
}

// ---- kernel A: generate -----------------------------------------------------------------------------------
// One thread per work item (sample, 8x4 pixel block, lane).  Camera ray (RayTracerProgram.cpp:133-165),
// then the shape list up to the first mesh whose bounds the ray enters.  A ray that ends there having
// hit nothing — most of them: they miss every bound and see the sky — is retired on the spot; the
// rest become paths: pool record + an entry in the round-0 queue, compacted per warp by ballot.
// VIEW: the camera rays of rt_gpu_render_view's turned camera (camera_ray_view), everything else unchanged.
// LIST: the pixels of a masked render: thread t takes work item a.list[t] of the *a.list_count the compaction kept
// (threads past the count idle), so "block" below is a group of 32 list entries; everything else unchanged.
template <bool CULL, int MODE, bool VIEW, bool LIST>
__device__ __forceinline__ void generate_items(const DevScene& sc, const RenderArgs& a, const WaveArgs& w, const ViewBasis& view)
{
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    // One thread per PIXEL of the work list (8x4 block, lane), looping over the chunk's samples: the
    // pixel decode, the base direction and the pixel half of the RNG key are computed once.  Grid-stride,
    // whole warps together (the queue pushes want converged lanes).  A retry pass instead takes one
    // turned-away item per thread.
    const unsigned stride = gridDim.x * blockDim.x;
    const bool retry = w.retry_in != nullptr;
    const unsigned nthreads_needed = retry ? (*w.retry_in_count < w.item_count ? *w.retry_in_count : w.item_count)
                                           : LIST ? *a.list_count : a.num_blocks * 32u;
    if (nthreads_needed == 0) return;
    const unsigned rounded = (nthreads_needed + 31u) & ~31u;
    const int sample_count = retry ? 1 : a.num_samples;
    const size_t frame = (size_t)a.width * a.height;
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < rounded; t += stride)
    {
        unsigned bl = 0, first_sample = 0;
        int lane_in_block = 0, px = -1, cx = 0, cy = 0;
        if (t < nthreads_needed)
        {
            if (retry)
            {
                const unsigned item = w.retry_in[t];
                const unsigned blk = item >> 5;
                first_sample = blk / a.num_blocks;
                bl = blk - first_sample * a.num_blocks;
                lane_in_block = (int)(item & 31u);
            }
            else { bl = t >> 5; lane_in_block = (int)(t & 31u); }
            if (LIST)
            {
                const unsigned item = a.list[(bl << 5) | (unsigned)lane_in_block];
                px = block_pixel(a, item >> 5, (int)(item & 31u), cx, cy);
            }
            else px = block_pixel(a, bl, lane_in_block, cx, cy);
        }
        float base_dx = 0.0f, base_dy = 0.0f;
        camera_base(a.width, a.height, cx, cy, base_dx, base_dy);
        const uint32_t pixel_key = rt_rng_key_pixel(a.seed, (uint32_t)px);
        // when every shape has culling bounds, a ray that misses them all needs no query state at all
        const bool all_bounded = a.all_bounded != 0;
        float3 b0min = V3(0, 0, 0), b0max = V3(0, 0, 0);
        if (all_bounded && sc.num_shapes > 0) { b0min = ld3(sc.shapes[0].bounds_min); b0max = ld3(sc.shapes[0].bounds_max); }
        // sky samples of the current pass that were retired in place (a thread meets a pass's four sub-samples in order)
        const bool fold_sky = a.antialias && !retry && (MODE == RT_MODE_PATH || MODE == RT_MODE_PREVIEW);
        unsigned sky_mask = 0u;
        float sky_y0 = 0.0f, sky_y1 = 0.0f, sky_y2 = 0.0f, sky_y3 = 0.0f;
        for (int k = 0; k < sample_count; k++)
        {
            const unsigned smp = first_sample + (unsigned)k;
            bool live = false;
            Query q;
            PathState s;
            int state = ST_IDLE;
            const Counters before = cnt;
            if (px >= 0)
            {
                s.pixel = px; s.slot = (int)smp;
                // spp is 4 (antialias) or 1
                const int pass = a.pass_begin + (a.antialias ? (int)(smp >> 2) : (int)smp);
                const int sub = a.antialias ? (int)(smp & 3u) : -1;
                s.rng.key = rt_rng_key_sample(pixel_key, (uint32_t)(a.antialias ? pass * 4 + sub : pass));
                s.rng.n = 0;
                const Ray cam = VIEW ? camera_ray_view(sc, view, a.width, base_dx, base_dy, RT_PRIMARY_LIKE(MODE) ? -1 : sub, s.rng)
                                     : camera_ray_from_base(sc, a.width, base_dx, base_dy, RT_PRIMARY_LIKE(MODE) ? -1 : sub, s.rng);
                cnt.camera_rays++;
                s.depth_left = a.max_bounce; s.sp = 0; s.pass_mask = 0; s.light = 0; s.seg_dist = cam.dist;
                s.w_pos = s.w_nrm = s.w_surface = s.w_sum = V3(0, 0, 0);
                if ((MODE == RT_MODE_PATH || MODE == RT_MODE_PREVIEW) && a.max_bounce == 0)
                    a.samples[(size_t)s.slot * frame + s.pixel] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                else
                {
                    bool enters = !all_bounded;
                    if (all_bounded)
                    {
                        // FindIntersectionWithScene's bounds tests only (RayTracerScene.cpp:107-110)
                        const RayPre pre = ray_pre(cam);
                        float tlo, thi;
                        for (int si = 0; si < sc.num_shapes && !enters; si++)
                            enters = si == 0 ? slab_general(cam, pre, b0min, b0max, tlo, thi)
                                             : slab_general(cam, pre, ld3(sc.shapes[si].bounds_min), ld3(sc.shapes[si].bounds_max), tlo, thi);
                    }
                    if (!enters)
                    {
                        cnt.rays++;
                        cnt.node_visits += (unsigned)sc.num_shapes;
                        state = ST_SHADE;
                        q.hit_shape = -1;
                    }
                    else
                    {
                        query_begin(q, cam, false, cnt);
                        state = ST_SHAPES;
                        query_shapes<CULL>(sc, q, state, cnt);
                    }
                    live = true;
                    if (state == ST_SHADE && q.hit_shape == -1)
                    {
                        // nothing hit and no mesh to walk: RayTrace's miss branch (RayTracerScene.cpp:90-94)
                        if (RT_PRIMARY_LIKE(MODE))
                        {
                            a.prim_ids[s.pixel] = make_int2(-1, -1);
                            a.prim_dist[s.pixel] = 0.0f;
                            if (MODE == RT_MODE_GUIDES) a.guide[s.pixel] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        }
                        else if (fold_sky)
                        {
                            // held back until the pass's fourth sub-sample: a pixel whose four camera rays all see
                            // the sky (most pixels of most frames) writes ONE folded colour instead of four samples
                            // (the sky colour is a function of the direction's y alone, so that is all that is kept)
                            if (sub == 0) sky_y0 = cam.d.y; else if (sub == 1) sky_y1 = cam.d.y; else if (sub == 2) sky_y2 = cam.d.y; else sky_y3 = cam.d.y;
                            sky_mask |= 1u << sub;
                        }
                        else
                        {
                            const float3 L = sky_color(cam.d);
                            a.samples[(size_t)s.slot * frame + s.pixel] = make_float4(L.x, L.y, L.z, 0.0f);
                        }
                        live = false;
                    }
                }
            }
            if (fold_sky && (smp & 3u) == 3u && sky_mask != 0u)
            {
                float4* const slot0 = a.samples + (size_t)(smp - 3u) * frame + px;
                const float3 up = V3(0.0f, 0.0f, 0.0f);
                if (sky_mask == 15u)
                {
                    // ThreadWorker_Render's c = 0; c += RayTrace(..) x 4; c /= 4 (RayTracerProgram.cpp:144-169), here rather
                    // than in the fold kernel; .w = 1 tells that kernel the pass colour is ready (samples carry .w = 0)
                    float3 c = V3(0.0f, 0.0f, 0.0f);
                    c = add3(c, sky_color(V3(up.x, sky_y0, up.z)));
                    c = add3(c, sky_color(V3(up.x, sky_y1, up.z)));
                    c = add3(c, sky_color(V3(up.x, sky_y2, up.z)));
                    c = add3(c, sky_color(V3(up.x, sky_y3, up.z)));
                    slot0[0] = make_float4(c.x / 4.0f, c.y / 4.0f, c.z / 4.0f, 1.0f);
                }
                else
                {
                    if (sky_mask & 1u) { const float3 L = sky_color(V3(up.x, sky_y0, up.z)); slot0[0] = make_float4(L.x, L.y, L.z, 0.0f); }
                    if (sky_mask & 2u) { const float3 L = sky_color(V3(up.x, sky_y1, up.z)); slot0[frame] = make_float4(L.x, L.y, L.z, 0.0f); }
                    if (sky_mask & 4u) { const float3 L = sky_color(V3(up.x, sky_y2, up.z)); slot0[2 * frame] = make_float4(L.x, L.y, L.z, 0.0f); }
                    if (sky_mask & 8u) { const float3 L = sky_color(V3(up.x, sky_y3, up.z)); slot0[3 * frame] = make_float4(L.x, L.y, L.z, 0.0f); }
                }
                sky_mask = 0u;
            }
            // round 0's queue is the identity: path id == queue position, one atomic per warp
            unsigned spare = 0xffffffffu;
            const unsigned id = w.packets ? path_alloc_packet(w.counts + 0, live, spare) : path_alloc(w.counts + 0, live);
            const bool full = live && id >= w.pool.cap;
            if (spare < w.pool.cap)
            {
                // filler of a packet: an entry every kernel skips
                w.pool.cur[spare] = make_int4(0, -1, ST_IDLE, 0);
                w.queue[0][spare] = spare;
            }
            if (live && !full)
            {
                // a camera ray whose only remaining chance is this last mesh: if the walk finds nothing the
                // walk kernel itself retires it with the sky colour (no trip through the shade kernel)
                const bool sky_on_miss = (MODE == RT_MODE_PATH || MODE == RT_MODE_PREVIEW) && state == ST_TRAVERSE &&
                                         q.hit_shape == -1 && q.si == sc.num_shapes - 1;
                pool_store<MODE>(w.pool, id, q, state, s, sky_on_miss);
                w.queue[0][id] = id;
            }
            // pool full: the item is turned away untouched (its counters too) and generated again by the retry pass
            if (full) cnt = before;
            queue_push(w.retry_out, w.retry_out_count, full, ((smp * a.num_blocks + bl) << 5) | (unsigned)lane_in_block);
        }
    }
    flush_counters(cnt, a.counters, a.exact);
}

template <bool CULL, int MODE>
__global__ void __launch_bounds__(256, RT_GEN_BLOCKS)
rt_generate_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w)
{
    generate_items<CULL, MODE, false, false>(sc, a, w, ViewBasis());
}

template <bool CULL, int MODE>
__global__ void __launch_bounds__(256, RT_GEN_BLOCKS)
rt_generate_view_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w, const ViewBasis view)
{
    generate_items<CULL, MODE, true, false>(sc, a, w, view);
}

// rt_gpu_render_masked: the generate kernels above over the compacted pixel list (VIEW: with a turned camera)
template <bool CULL, int MODE, bool VIEW>
__global__ void __launch_bounds__(256, RT_GEN_BLOCKS)
rt_generate_list_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w, const ViewBasis view)
{
    generate_items<CULL, MODE, VIEW, true>(sc, a, w, view);
}

// ---- kernel Q: generate for a batch of ray queries (rt_gpu_query_rays) ---------------------------------------------
// What rt_generate_kernel does up to its queue push, for the caller's rays: one thread per ray (grid-stride, whole
// warps together), the shape list up to the first mesh whose bounds the ray enters.  A query that needs no walk — it
// missed everything, hit only analytic shapes, or an analytic shape occluded it — writes its result on the spot; the
// rest become pool records (pa.x = the ray's place in the batch) in round 0, allocated in packets of 32 so that a
// round-0 packet is 32 consecutive rays of the caller's order.  The host hands a batch over in pieces that fit the
// pool: no item is ever turned away here.
// Radiance queries (rt_gpu_radiance_rays, MODE = RT_MODE_PATH / PREVIEW / WHITTED) start a whole path instead, as
// rt_generate_kernel does after its camera ray: the ray's own RNG stream, the bounce budget, the sky on the spot for
// a ray that hit nothing and has no mesh to walk, and a round-0 record for every other ray (analytic hits included:
// the shade kernel shades them).  The sample of ray i is a.samples[i] (the host points it at the caller's rgba).
template <bool CULL, int MODE>
__global__ void __launch_bounds__(256, 2)
rt_query_generate_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w)
{
    constexpr bool radiance = MODE == RT_MODE_PATH || MODE == RT_MODE_PREVIEW || MODE == RT_MODE_WHITTED;
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    const unsigned n = (unsigned)a.q_count;
    const unsigned rounded = (n + 31u) & ~31u;
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < rounded; t += stride)
    {
        bool live = false;
        Query q;
        PathState s;
        int state = ST_IDLE;
        if (t < n)
        {
            const float* p = a.q_rays + 7 * (size_t)t;
            Ray r; r.o = V3(p[0], p[1], p[2]); r.d = V3(p[3], p[4], p[5]); r.dist = p[6];
            s.pixel = (int)t; s.slot = 0;
            s.depth_left = 0; s.sp = 0; s.pass_mask = 0; s.light = 0; s.seg_dist = r.dist;
            if (radiance)
            {
                const uint32_t stream_id = a.q_stream ? a.q_stream[t] : a.q_stream_base + t;
                s.rng.key = rt_rng_key(a.seed, stream_id, a.q_sample); s.rng.n = a.q_first_draw;
                s.depth_left = a.max_bounce;
                s.w_pos = s.w_nrm = s.w_surface = s.w_sum = V3(0, 0, 0);
                // RayTrace(ray, 0) returns black before any query (RayTracerScene.cpp:39-42)
                if (MODE != RT_MODE_WHITTED && a.max_bounce == 0) a.samples[t] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                else
                {
                    query_begin(q, r, false, cnt);
                    state = ST_SHAPES;
                    query_shapes<CULL>(sc, q, state, cnt);
                    live = true;
                    if (state == ST_SHADE && q.hit_shape == -1)
                    {
                        // nothing hit and no mesh to walk: RayTrace's miss branch (RayTracerScene.cpp:90-94)
                        const float3 L = sky_color(r.d);
                        a.samples[t] = make_float4(L.x, L.y, L.z, 0.0f);
                        live = false;
                    }
                }
            }
            else
            {
                query_begin(q, r, MODE == RT_QMODE_ANY, cnt);
                state = ST_SHAPES;
                query_shapes<CULL>(sc, q, state, cnt);
                live = state == ST_TRAVERSE;
                if (!live) query_result<MODE>(a, (int)t, q);
                s.rng.key = 0; s.rng.n = 0;
            }
        }
        unsigned spare = 0xffffffffu;
        const unsigned id = path_alloc_packet(w.counts + 0, live, spare);
        if (spare < w.pool.cap)
        {
            // filler of a packet: an entry every kernel skips
            w.pool.cur[spare] = make_int4(0, -1, ST_IDLE, 0);
            w.queue[0][spare] = spare;
        }
        if (live)
        {
            // (rt_generate_kernel's rule: a path ray whose only remaining chance is this last mesh is retired with the
            // sky colour by the walk kernel itself if the walk finds nothing)
            const bool sky_on_miss = (MODE == RT_MODE_PATH || MODE == RT_MODE_PREVIEW) && state == ST_TRAVERSE &&
                                     q.hit_shape == -1 && q.si == sc.num_shapes - 1;
            pool_store<MODE>(w.pool, id, q, state, s, sky_on_miss);
            w.queue[0][id] = id;
        }
    }
    flush_counters(cnt, a.counters, a.exact);
}

// ---- kernel T: walk ------------------------------------------------------------------------------------------
// Persistent warps.  A lane pops a path id from the round's queue, loads the ray, and walks the mesh its
// shape cursor points at — KdNode::TestRayIntersection (KdTree.cpp:128-195) on the pre-order,
// escape-threaded node array, see rt_device.cuh — to the end; then it stores (best leaf, position,
// shrunken Distance) and pops the next id, so a warp's 32 lanes stay on walks of their own length.
// Rounds of "node steps until the walking lanes hold a leaf, then those triangle tests together".
template <bool CULL>
__global__ void __launch_bounds__(256, RT_WALK_BLOCKS)
rt_walk_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w, int round, int resumed)
{
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    // resumed: the walks the packet kernel handed back (they continue at their cursor); else the round's queue
    const unsigned round_count = w.counts[round] < w.pool.cap ? w.counts[round] : w.pool.cap;
    const unsigned count = resumed ? w.scounts[round] : round_count;
    const unsigned* __restrict__ queue = resumed ? w.slowq : w.queue[round & 1];
    unsigned* head = resumed ? w.sheads + round : w.heads + round;
    if (count == 0 || round_count < w.small_round) return;   // empty, or thin: the long-walk kernel takes all of it
    const unsigned long_limit = round_count < w.thin_count ? w.thin_limit : w.long_limit;
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    unsigned win_pos = 0, win_end = 0;
    bool exhausted = count == 0;

    bool have = false;
    unsigned id = 0;
    Ray r; r.o = V3(0, 0, 0); r.d = V3(0, 0, 1); r.dist = 0.0f;
    RayPre pre = ray_pre(r);
    bool any = false, weird = false, wide = false, sky_on_miss = false;
    float3 pad3 = V3(0, 0, 0);
    float growth = 0.0f;
    const float4* __restrict__ nodes = nullptr;
    const float4* __restrict__ tris = nullptr;
    int n = 0, i = 0, best = -1;
    float3 bpos = V3(0, 0, 0);
    unsigned nodes_seen = 0, tris_seen = 0;
    unsigned walk_start = 0, walk_max = 0;

    for (;;)
    {
        // ---- refill: lanes without a walk pop ids (ballot -> rank -> window item) ----------------------
        for (;;)
        {
            const unsigned idle = __ballot_sync(RT_FULL_MASK, !have);
            if (idle == 0) break;
            if (win_pos >= win_end)
            {
                if (exhausted) break;
                unsigned base = 0;
                if (lane == 0) base = atomicAdd(head, w.window);
                base = __shfl_sync(RT_FULL_MASK, base, 0);
                if (base >= count) { exhausted = true; break; }
                win_pos = base;
                win_end = count - base < w.window ? count : base + w.window;
            }
            const unsigned item = win_pos + (unsigned)__popc(idle & lt_mask);
            if (!have && item < win_end)
            {
                id = queue[item];
                const int4 cur = w.pool.cur[id];
                if ((cur.z & 255) == ST_TRAVERSE)
                {
                    const float4 ro = w.pool.ro[id], rd = w.pool.rd[id];
                    r.o = xyz(ro); r.dist = ro.w; r.d = xyz(rd);
                    pre = ray_pre(r);
                    weird = !(pre.ex && pre.ey && pre.ez && finite3(r.o) && finite3(r.d));
                    any = (cur.z & 256) != 0;
                    sky_on_miss = (cur.z & 512) != 0;
                    const DevMesh* m = sc.meshes + sc.shapes[cur.x].mesh;
                    nodes = m->nodes; tris = m->tris; n = m->num_nodes;
                    if (CULL)
                    {
                        pre.cull_pad = cull_pad_for(r, pre, m->cull_scale);
                        growth = cull_growth(r, m->cull_scale);
                        // a disabled axis is not constrained (inv = 0 there: its interval is [-pad, pad] around 0)
                        pad3.x = pre.ex ? growth * fabsf(pre.inv.x) + growth : FLT_MAX;
                        pad3.y = pre.ey ? growth * fabsf(pre.inv.y) + growth : FLT_MAX;
                        pad3.z = pre.ez ? growth * fabsf(pre.inv.z) + growth : FLT_MAX;
                        const bool finite = finite3(r.o) && finite3(r.d) && pre.cull_pad < FLT_MAX;
                        wide = finite && (pre.cull_pad > 4096.0f * growth || !(pre.ex && pre.ey && pre.ez));    // |d| < 2.4e-4 on some axis
                    }
                    i = 0; best = -1; bpos = V3(0, 0, 0);
                    if (resumed)
                    {
                        const float4 bp = w.pool.bp[id];
                        i = __float_as_int(bp.w); best = cur.y; bpos = xyz(bp);
                    }
                    walk_start = nodes_seen;
                    have = true;
                }
            }
            const unsigned taken = win_pos + (unsigned)__popc(idle);
            win_pos = taken < win_end ? taken : win_end;
        }
        if (__ballot_sync(RT_FULL_MASK, have) == 0) break;

        // ---- walk until too few lanes are left walking ---------------------------------------------------
        const bool verbatim = __any_sync(RT_FULL_MASK, have && weird);
        const bool widewarp = CULL && __any_sync(RT_FULL_MASK, have && wide);
        const int min_lanes = exhausted ? 1 : w.min_lanes;
        for (;;)
        {
            // Node phase.  The leaves a walk reaches do not depend on the hits it has accepted (the
            // reference's box test is a line test, KdTree.cpp:131; the culling above only drops leaves
            // that would be rejected anyway), so a lane that has found a leaf keeps walking to its NEXT
            // leaf while its neighbours are still looking for their first: up to two leaves are held and
            // then tested in walk order.  Fewer lanes wait, and the triangle phase runs fuller.
            int leaf[RT_LEAF_SLOTS];
#pragma unroll
            for (int k = 0; k < RT_LEAF_SLOTS; k++) leaf[k] = -1;
            for (;;)
            {
                const unsigned stepping = __ballot_sync(RT_FULL_MASK, have && leaf[RT_LEAF_SLOTS - 1] < 0 && i < n);
                if (stepping == 0) break;
                if (w.leaf_wait > 0 && __popc(stepping) < w.leaf_wait &&
                    __ballot_sync(RT_FULL_MASK, leaf[0] >= 0) != 0) break;
                // a few node steps per vote (RT_STEPS_PER_VOTE): the loop control above costs as much as half a step
#pragma unroll
                for (int u = 0; u < RT_STEPS_PER_VOTE; u++)
                {
                    if (have && leaf[RT_LEAF_SLOTS - 1] < 0 && i < n)
                    {
                        float4 na, nb;
                        ld32(nodes + 2 * (size_t)i, na, nb);
                        const int escape = __float_as_int(na.w);
                        const int tri = __float_as_int(nb.w);
                        nodes_seen++;
                        float tlo, thi;
                        bool enter = verbatim ? slab_general(r, pre, xyz(na), xyz(nb), tlo, thi)
                                              : slab_fast(r, pre, xyz(na), xyz(nb), tlo, thi);
                        if (CULL)
                        {
                            if (widewarp && wide) enter = enter && !cull_axes(r, pre, pad3, xyz(na), xyz(nb), r.dist * 1.0078125f + growth, growth);
                            else enter = enter && !(thi < -pre.cull_pad) && !(tlo > r.dist * 1.0078125f + pre.cull_pad);
                        }
                        if (!enter) i = escape;
                        else if (tri < 0) i = i + 1;
                        else
                        {
                            bool placed = false;
#pragma unroll
                            for (int k = 0; k < RT_LEAF_SLOTS; k++)
                                if (!placed && leaf[k] < 0) { leaf[k] = tri; placed = true; }
                            i = escape;
                        }
                    }
                }
            }
            // Triangle phase: the held leaves, in walk order
#pragma unroll
            for (int k = 0; k < RT_LEAF_SLOTS; k++)
            {
                const int lf = leaf[k];
                if (__ballot_sync(RT_FULL_MASK, lf >= 0) == 0) break;
                if (lf >= 0)
                {
                    float4 t0, t1, t2, t3;
                    ld32(tris + 4 * (size_t)lf, t0, t1);
                    ld32(tris + 4 * (size_t)lf + 2, t2, t3);
                    tris_seen++;
                    float3 hp; float hd;
                    if (triangle_test(r, xyz(t0), xyz(t1), xyz(t2), xyz(t3), hp, hd))
                    {
                        r.dist = hd;
                        bpos = hp;
                        best = lf;
                        if (CULL && any)
                        {
                            i = n;
#pragma unroll
                            for (int j = 0; j < RT_LEAF_SLOTS; j++) leaf[j] = -1;
                        }
                    }
                }
            }
            if (have && i >= n)
            {
                // walk complete: hand the result to the shade kernel
                int* cur = reinterpret_cast<int*>(w.pool.cur + id);
                if (best < 0 && sky_on_miss)
                {
                    // RayTrace's miss branch (RayTracerScene.cpp:90-94) for a camera ray: nothing to fold
                    const int4 pa = w.pool.pa[id];
                    const float3 L = sky_color(r.d);
                    a.samples[(size_t)pa.y * ((size_t)a.width * a.height) + pa.x] = make_float4(L.x, L.y, L.z, 0.0f);
                    cur[2] = ST_IDLE;           // the shade kernel skips it
                }
                else
                {
                    w.pool.ro[id].w = r.dist;
                    cur[1] = best;
                    cur[2] = ST_MESHDONE | (any ? 256 : 0);
                    if (best >= 0) w.pool.bp[id] = make_float4(bpos.x, bpos.y, bpos.z, 0.0f);
                }
                walk_max = max(walk_max, nodes_seen - walk_start);
                have = false;
            }
            else if (have && nodes_seen - walk_start > long_limit)
            {
                // A walk this long would hold the round: park it (cursor, best hit so far) for the
                // long-walk kernel, which spends a whole warp on it.  No leaf is pending here.
                w.pool.ro[id].w = r.dist;
                reinterpret_cast<int*>(w.pool.cur + id)[1] = best;
                w.pool.bp[id] = make_float4(bpos.x, bpos.y, bpos.z, __int_as_float(i));
                w.longq[atomicAdd(w.lcounts + round, 1u)] = id;
                have = false;
            }
            if (__popc(__ballot_sync(RT_FULL_MASK, have)) < min_lanes) break;
        }
    }
    cnt.node_visits = nodes_seen; cnt.tri_visits = tris_seen;
    flush_counters(cnt, a.counters, a.exact);
    // longest single walk of the batch (tooling: rt_gpu_debug_rounds)
    for (int o = 16; o > 0; o >>= 1) walk_max = max(walk_max, __shfl_xor_sync(RT_FULL_MASK, walk_max, o));
    if (lane == 0 && walk_max > 0) atomicMax(w.counts + RT_MAX_ROUNDS, walk_max);
}

// ---- kernel P: packet walk (coherent rounds) ---------------------------------------------------------------
// Round 0 holds camera rays in generation order: 32 consecutive entries come from one 8x4-pixel block, so
// their walks visit almost the same nodes.  Here a warp walks its 32 rays TOGETHER: one cursor per lane as
// before, but each step the warp visits the smallest cursor c of its lanes — the array is in visiting
// order, so every lane still meets exactly its own nodes, in its own order — loads node c ONCE (uniform
// address: one transaction instead of up to 32), and the lanes standing at c test it.  A leaf is tested on
// the spot by the lanes that entered its box (same triangle for all of them).  Per ray the tests, their
// order and their results are those of rt_walk_kernel; only the schedule differs.  The warp needs |union of
// the lanes' node sets| steps instead of sum/active-lanes, without divergence and with far fewer memory
// requests.  Lanes of other meshes wait their turn (one group per mesh); a packet that exceeds the step
// budget parks its unfinished lanes for the long-walk kernel.
template <bool CULL>
__global__ void __launch_bounds__(256, RT_WALK_BLOCKS)
rt_walk_packet_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w, int round)
{
    const int lane = threadIdx.x & 31;
    const unsigned count = w.counts[round] < w.pool.cap ? w.counts[round] : w.pool.cap;
    const unsigned* __restrict__ queue = w.queue[round & 1];
    unsigned* head = w.heads + round;
    if (count == 0 || count < w.small_round) return;   // empty, or thin: the long-walk kernel takes all of it
    const unsigned step_limit = count < w.thin_count ? w.thin_limit : w.long_limit;
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    unsigned nodes_seen = 0, tris_seen = 0;
    for (;;)
    {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(head, 32u);
        base = __shfl_sync(RT_FULL_MASK, base, 0);
        if (base >= count) break;
        const unsigned item = base + (unsigned)lane;
        unsigned id = 0;
        bool active = false;
        int shape = -1;
        bool any = false, sky_on_miss = false;
        Ray r; r.o = V3(0, 0, 0); r.d = V3(0, 0, 1); r.dist = 0.0f;
        if (item < count)
        {
            id = queue[item];
            const int4 cur = w.pool.cur[id];
            if ((cur.z & 255) == ST_TRAVERSE)
            {
                const float4 ro = w.pool.ro[id], rd = w.pool.rd[id];
                r.o = xyz(ro); r.dist = ro.w; r.d = xyz(rd);
                any = (cur.z & 256) != 0;
                sky_on_miss = (cur.z & 512) != 0;
                shape = cur.x;
                active = true;
            }
        }
        RayPre pre = ray_pre(r);
        const bool weird = !(pre.ex && pre.ey && pre.ez && finite3(r.o) && finite3(r.d));
        unsigned todo = __ballot_sync(RT_FULL_MASK, active);
        while (todo != 0)
        {
            // one group per mesh (a scene with one mesh: one group)
            const int leader = __ffs((int)todo) - 1;
            const int gshape = __shfl_sync(RT_FULL_MASK, shape, leader);
            const bool mine = active && shape == gshape;
            todo &= ~__ballot_sync(RT_FULL_MASK, mine);
            const DevMesh* m = sc.meshes + sc.shapes[gshape].mesh;
            const float4* __restrict__ nodes = m->nodes;
            const float4* __restrict__ tris = m->tris;
            const int n = m->num_nodes;
            float3 pad3 = V3(0, 0, 0);
            float growth = 0.0f;
            bool wide = false;
            if (CULL)
            {
                pre.cull_pad = cull_pad_for(r, pre, m->cull_scale);
                growth = cull_growth(r, m->cull_scale);
                pad3.x = pre.ex ? growth * fabsf(pre.inv.x) + growth : FLT_MAX;
                pad3.y = pre.ey ? growth * fabsf(pre.inv.y) + growth : FLT_MAX;
                pad3.z = pre.ez ? growth * fabsf(pre.inv.z) + growth : FLT_MAX;
                const bool finite = finite3(r.o) && finite3(r.d) && pre.cull_pad < FLT_MAX;
                wide = finite && (pre.cull_pad > 4096.0f * growth || !(pre.ex && pre.ey && pre.ez));
            }
            const bool verbatim = __any_sync(RT_FULL_MASK, mine && weird);
            const bool widewarp = CULL && __any_sync(RT_FULL_MASK, mine && wide);
            int best = -1;
            float3 bpos = V3(0, 0, 0);
            unsigned cursor = mine ? 0u : 0xffffffffu;
            const unsigned group_lanes = (unsigned)__popc(__ballot_sync(RT_FULL_MASK, mine));
            unsigned steps = 0;
            bool parked = false, done = false;
            while (!done)
            {
                // a window of packet_probe steps, then the packet is judged
                const unsigned seen_before = nodes_seen;
                for (unsigned k = 0; k < w.packet_probe; k++)
                {
                    const unsigned c = __reduce_min_sync(RT_FULL_MASK, cursor);
                    if (c >= (unsigned)n) { done = true; break; }
                    float4 na, nb;
                    ld32(nodes + 2 * (size_t)c, na, nb);
                    const int escape = __float_as_int(na.w);
                    const int tri = __float_as_int(nb.w);
                    bool enter = false;
                    if (cursor == c)
                    {
                        nodes_seen++;
                        float tlo, thi;
                        enter = verbatim ? slab_general(r, pre, xyz(na), xyz(nb), tlo, thi)
                                         : slab_fast(r, pre, xyz(na), xyz(nb), tlo, thi);
                        if (CULL)
                        {
                            if (widewarp && wide) enter = enter && !cull_axes(r, pre, pad3, xyz(na), xyz(nb), r.dist * 1.0078125f + growth, growth);
                            else enter = enter && !(thi < -pre.cull_pad) && !(tlo > r.dist * 1.0078125f + pre.cull_pad);
                        }
                        cursor = (enter && tri < 0) ? c + 1u : (unsigned)escape;
                    }
                    if (tri >= 0 && __any_sync(RT_FULL_MASK, enter))
                    {
                        float4 t0, t1, t2, t3;
                        ld32(tris + 4 * (size_t)tri, t0, t1);
                        ld32(tris + 4 * (size_t)tri + 2, t2, t3);
                        if (enter)
                        {
                            tris_seen++;
                            float3 hp; float hd;
                            if (triangle_test(r, xyz(t0), xyz(t1), xyz(t2), xyz(t3), hp, hd))
                            {
                                r.dist = hd; bpos = hp; best = tri;
                                if (CULL && any) cursor = (unsigned)n;
                            }
                        }
                    }
                }
                if (done) break;
                steps += w.packet_probe;
                // Not a coherent packet after all (rays of one pixel block spread over many small triangles): the
                // steps of the last window were mostly other lanes' nodes (the top of the tree is common to all
                // rays; coherence shows, or ends, further down).  Its unfinished lanes go on one by one in
                // rt_walk_kernel, from where they are.  Likewise a packet that outlasts the step budget: those
                // lanes go on alone in the long-walk kernel.
                const unsigned tests = __reduce_add_sync(RT_FULL_MASK, nodes_seen - seen_before);
                const bool incoherent = tests * 32u < w.packet_probe * w.packet_min_lanes * group_lanes;
                if (incoherent || steps > step_limit)
                {
                    if (mine && cursor < (unsigned)n)
                    {
                        w.pool.ro[id].w = r.dist;
                        reinterpret_cast<int*>(w.pool.cur + id)[1] = best;
                        w.pool.bp[id] = make_float4(bpos.x, bpos.y, bpos.z, __int_as_float((int)cursor));
                        if (incoherent) w.slowq[atomicAdd(w.scounts + round, 1u)] = id;
                        else w.longq[atomicAdd(w.lcounts + round, 1u)] = id;
                        parked = true;
                    }
                    break;
                }
            }
            if (mine && !parked)
            {
                // walk complete: hand the result to the shade kernel
                int* curw = reinterpret_cast<int*>(w.pool.cur + id);
                if (best < 0 && sky_on_miss)
                {
                    const int4 pa = w.pool.pa[id];
                    const float3 L = sky_color(r.d);
                    a.samples[(size_t)pa.y * ((size_t)a.width * a.height) + pa.x] = make_float4(L.x, L.y, L.z, 0.0f);
                    curw[2] = ST_IDLE;
                }
                else
                {
                    w.pool.ro[id].w = r.dist;
                    curw[1] = best;
                    curw[2] = ST_MESHDONE | (any ? 256 : 0);
                    w.pool.bp[id] = make_float4(bpos.x, bpos.y, bpos.z, 0.0f);
                }
            }
        }
    }
    cnt.node_visits = nodes_seen; cnt.tri_visits = tris_seen;
    flush_counters(cnt, a.counters, a.exact);
}

// The device copy of an inner node keeps its right child in the `tri` field (-2 - index; any negative value
// still reads "inner node" to the sequential walks): right child = escape of the left child (k + 1).
__global__ void rt_patch_right_child(rt_bvh_node* nodes, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n && nodes[k].tri < 0) nodes[k].tri = -2 - (k + 1 < n ? nodes[k + 1].escape : n);
}

// ---- kernel L: long walks ------------------------------------------------------------------------------------
// One WARP per walk the walk kernel parked (or per entry of a thin round).  Two facts make a walk parallel
// without changing a bit of its result:
//   * which nodes a walk visits does not depend on what it hits (the reference's box test is a line test,
//     KdTree.cpp:131; culling with the Distance of the moment the walk was parked only drops leaves that
//     would be rejected anyway, Distance only shrinks), and
//   * the array is in visiting order, so "in the reference's order" == "by ascending leaf slot".
// So the warp first expands the rest of the tree as a FRONTIER — 32 pending nodes per step from a stack in
// shared memory, each lane one slab test, children pushed back (an inner node's `tri` field holds its right
// child, patched at upload) — collecting the leaves reached; then sorts those leaf slots and REPLAYS the
// triangle tests one after the other (Distance shrinks exactly as in the reference; every lane computes the
// same test on shuffled operands).  A 600-node walk is ~40 memory round trips instead of 600.
// The walk resumes at a cursor: the rest of the traversal is the cursor's subtree, then its escape's, ...;
// that chain is followed by lane 31, one link per step.  A frontier or leaf list that outgrows its shared
// memory falls back to the sequential window replay below (nothing has been written by then).
// The G lanes of a GROUP share one walk (G = 32, 16 or 8: a warp runs 1, 2 or 4 walks as independent
// mini-warps, every collective masked to the group).  A walk's frontier is rarely 32 nodes wide, and the
// kernel is bound by memory round trips, so narrower groups keep more walks in flight per SM.

// Sequential fallback: the next G nodes i..i+G-1 tested at once, the cursor replayed through the results.
template <bool CULL, int G>
__device__ __forceinline__ void longwalk_windows(const float4* __restrict__ nodes, const float4* __restrict__ tris, int n, int gl, unsigned gmask,
                                                 Ray& r, const RayPre& pre, float3 pad3, float growth, bool cull, bool any,
                                                 int& i, int& best, float3& bpos, unsigned& nodes_seen, unsigned& tris_seen)
{
    while (i < n)
    {
        const int node = i + gl;
        bool enter = false;
        int escape = n, tri = -1;
        if (node < n)
        {
            float4 na, nb;
            ld32(nodes + 2 * (size_t)node, na, nb);
            escape = __float_as_int(na.w); tri = __float_as_int(nb.w);
            float tlo, thi;
            enter = slab_general(r, pre, xyz(na), xyz(nb), tlo, thi);
            if (CULL && cull) enter = enter && !cull_axes(r, pre, pad3, xyz(na), xyz(nb), r.dist * 1.0078125f + growth, growth);
        }
        const int wend = i + G < n ? i + G : n;
        int c = i;
        while (c < wend)
        {
            const int src = c - i;
            const bool en = __shfl_sync(gmask, (int)enter, src, G) != 0;
            const int es = __shfl_sync(gmask, escape, src, G);
            const int tr = __shfl_sync(gmask, tri, src, G);
            nodes_seen++;
            if (!en) c = es;
            else if (tr < 0) c = c + 1;
            else
            {
                float4 t0, t1, t2, t3;
                ld32(tris + 4 * (size_t)tr, t0, t1);
                ld32(tris + 4 * (size_t)tr + 2, t2, t3);
                tris_seen++;
                float3 hp; float hd;
                c = es;
                if (triangle_test(r, xyz(t0), xyz(t1), xyz(t2), xyz(t3), hp, hd))
                {
                    r.dist = hd; bpos = hp; best = tr;
                    if (CULL && any) c = n;
                }
            }
        }
        i = c;
    }
}

template <bool CULL, int G>
__global__ void __launch_bounds__(256, RT_LONG_BLOCKS)
rt_longwalk_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w, int round)
{
    constexpr int CAP = RT_FW_INTS_PER_LANE * G;
    __shared__ int s_stack[256 * RT_FW_INTS_PER_LANE];
    __shared__ int s_leaf[256 * RT_FW_INTS_PER_LANE];
    const int lane = threadIdx.x & 31;
    const int gl = lane & (G - 1);                  // lane within the group
    const int gshift = lane - gl;
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << gshift);
    const unsigned lt_mask = (1u << gl) - 1u;
    int* stk = s_stack + (threadIdx.x / G) * CAP;
    int* lst = s_leaf + (threadIdx.x / G) * CAP;
    // a thin round (the walk kernel skipped it) is taken whole from the round's queue; otherwise only the
    // walks that kernel parked
    const unsigned round_count = w.counts[round] < w.pool.cap ? w.counts[round] : w.pool.cap;
    const bool whole = round_count < w.small_round;
    const unsigned count = whole ? round_count : w.lcounts[round];
    const unsigned* __restrict__ src = whole ? w.queue[round & 1] : w.longq;
    if (count == 0) return;
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    unsigned nodes_seen = 0, tris_seen = 0;
    for (;;)
    {
        unsigned e = 0;
        if (gl == 0) e = atomicAdd(w.lheads + round, 1u);
        e = __shfl_sync(gmask, e, 0, G);
        if (e >= count) break;
        const unsigned id = src[e];
        const int4 cur = w.pool.cur[id];
        if ((cur.z & 255) != ST_TRAVERSE) continue;      // (round 0 may hold entries that need no walk)
        // (a walk taken from the round's own queue has not begun: no cursor, no leaf; pool_store does not write bp)
        const float4 ro = w.pool.ro[id], rd = w.pool.rd[id], bp = whole ? make_float4(0.0f, 0.0f, 0.0f, 0.0f) : w.pool.bp[id];
        Ray r; r.o = xyz(ro); r.dist = ro.w; r.d = xyz(rd);
        RayPre pre = ray_pre(r);
        const bool any = (cur.z & 256) != 0, sky_on_miss = (cur.z & 512) != 0;
        const DevMesh* m = sc.meshes + sc.shapes[cur.x].mesh;
        const float4* __restrict__ nodes = m->nodes;
        const float4* __restrict__ tris = m->tris;
        const int n = m->num_nodes;
        float3 pad3 = V3(FLT_MAX, FLT_MAX, FLT_MAX);
        float growth = 0.0f;
        bool cull = false;
        if (CULL)
        {
            growth = cull_growth(r, m->cull_scale);
            pad3.x = pre.ex ? growth * fabsf(pre.inv.x) + growth : FLT_MAX;
            pad3.y = pre.ey ? growth * fabsf(pre.inv.y) + growth : FLT_MAX;
            pad3.z = pre.ez ? growth * fabsf(pre.inv.z) + growth : FLT_MAX;
            cull = finite3(r.o) && finite3(r.d) && growth < FLT_MAX && r.dist >= 0.0f;    // (see cull_pad_for)
        }
        int i = __float_as_int(bp.w), best = cur.y;
        float3 bpos = xyz(bp);
        const unsigned walk_start_seen = nodes_seen;

        // ---- frontier: the leaves the rest of the walk reaches -------------------------------------------
        const float reach = r.dist * 1.0078125f + growth;        // Distance at parking time: only shrinks from here
        int size = 0, nleaf = 0, chain = i;
        unsigned frontier_nodes = 0;
        bool overflow = false;
        while (size > 0 || chain < n)
        {
            const bool has_chain = chain < n;
            const int room = CAP - size;
            if (room < 4) { overflow = true; break; }
            // a popped node nets at most one entry (two children pushed), the chain node two
            int k = size < G - 1 ? size : G - 1;
            if (k + 2 > room) k = room - 2;
            int node = -1;
            if (gl < k) node = stk[size - 1 - gl];
            else if (gl == G - 1 && has_chain) node = chain;
            if (node >= n) node = -1;
            size -= k;
            __syncwarp(gmask);
            bool enter = false;
            int escape = n, tri = -1;
            if (node >= 0)
            {
                float4 na, nb;
                ld32(nodes + 2 * (size_t)node, na, nb);
                escape = __float_as_int(na.w); tri = __float_as_int(nb.w);
                float tlo, thi;
                enter = slab_general(r, pre, xyz(na), xyz(nb), tlo, thi);
                if (CULL && cull) enter = enter && !cull_axes(r, pre, pad3, xyz(na), xyz(nb), reach, growth);
            }
            frontier_nodes += (unsigned)__popc(__ballot_sync(gmask, node >= 0));
            if (has_chain) chain = __shfl_sync(gmask, escape, G - 1, G);
            const unsigned leaves = __ballot_sync(gmask, enter && tri >= 0) >> gshift;
            if (leaves != 0)
            {
                if (nleaf + __popc(leaves) > CAP) { overflow = true; break; }
                if (enter && tri >= 0) lst[nleaf + __popc(leaves & lt_mask)] = tri;
                nleaf += __popc(leaves);
            }
            const unsigned inner = __ballot_sync(gmask, enter && tri < 0) >> gshift;
            if (enter && tri < 0)
            {
                const int right = -2 - tri;
                const int pos = size + 2 * __popc(inner & lt_mask);
                // (right child on the bottom: the left subtree is expanded first, which keeps the stack short)
                stk[pos] = right < escape ? right : n;
                stk[pos + 1] = node + 1 < escape ? node + 1 : n;
            }
            size += 2 * __popc(inner);
            __syncwarp(gmask);
            // entries that name no node (single-child nodes of a foreign tree) are dropped when popped
            while (size > 0 && stk[size - 1] >= n) size--;
        }
        if (overflow)
        {
            __syncwarp(gmask);
            longwalk_windows<CULL, G>(nodes, tris, n, gl, gmask, r, pre, pad3, growth, cull, any, i, best, bpos, nodes_seen, tris_seen);
        }
        else
        {
            nodes_seen += frontier_nodes;
            // ---- replay: sort the leaf slots (== visiting order), then the triangle tests in that order ----
            __syncwarp(gmask);
            for (int x = gl; x < nleaf; x += G)
            {
                const int v = lst[x];
                int rank = 0;
                for (int j = 0; j < nleaf; j++) rank += lst[j] < v ? 1 : 0;
                stk[rank] = v;
            }
            __syncwarp(gmask);
            bool stop = false;
            for (int base = 0; base < nleaf && !stop; base += G)
            {
                const int lf = base + gl < nleaf ? stk[base + gl] : -1;
                float4 t0 = make_float4(0, 0, 0, 0), t1 = t0, t2 = t0, t3 = t0;
                if (lf >= 0)
                {
                    ld32(tris + 4 * (size_t)lf, t0, t1);
                    ld32(tris + 4 * (size_t)lf + 2, t2, t3);
                }
                const int batch = nleaf - base < G ? nleaf - base : G;
                for (int k = 0; k < batch; k++)
                {
                    const float3 p0 = V3(__shfl_sync(gmask, t0.x, k, G), __shfl_sync(gmask, t0.y, k, G), __shfl_sync(gmask, t0.z, k, G));
                    const float3 p1 = V3(__shfl_sync(gmask, t1.x, k, G), __shfl_sync(gmask, t1.y, k, G), __shfl_sync(gmask, t1.z, k, G));
                    const float3 p2 = V3(__shfl_sync(gmask, t2.x, k, G), __shfl_sync(gmask, t2.y, k, G), __shfl_sync(gmask, t2.z, k, G));
                    const float3 nn = V3(__shfl_sync(gmask, t3.x, k, G), __shfl_sync(gmask, t3.y, k, G), __shfl_sync(gmask, t3.z, k, G));
                    const int slot = __shfl_sync(gmask, lf, k, G);
                    tris_seen++;
                    float3 hp; float hd;
                    if (triangle_test(r, p0, p1, p2, nn, hp, hd))
                    {
                        r.dist = hd; bpos = hp; best = slot;
                        if (CULL && any) { stop = true; break; }
                    }
                }
            }
            __syncwarp(gmask);
        }
        if (gl == 0)
        {
            atomicMax(w.counts + RT_MAX_ROUNDS, nodes_seen - walk_start_seen);      // tooling: longest walk
            int* curw = reinterpret_cast<int*>(w.pool.cur + id);
            if (best < 0 && sky_on_miss)
            {
                const int4 pa = w.pool.pa[id];
                const float3 L = sky_color(r.d);
                a.samples[(size_t)pa.y * ((size_t)a.width * a.height) + pa.x] = make_float4(L.x, L.y, L.z, 0.0f);
                curw[2] = ST_IDLE;
            }
            else
            {
                w.pool.ro[id].w = r.dist;
                curw[1] = best;
                curw[2] = ST_MESHDONE | (any ? 256 : 0);
                w.pool.bp[id] = make_float4(bpos.x, bpos.y, bpos.z, 0.0f);
            }
        }
    }
    __syncwarp();
    // every lane of a group saw the same walk: count it once
    if (gl == 0) { cnt.node_visits = nodes_seen; cnt.tri_visits = tris_seen; }
    flush_counters(cnt, a.counters, a.exact);
}

// ---- kernel S: shade ----------------------------------------------------------------------------------------
// One thread per entry of the round's queue (grid-stride).  Finishes the mesh hit (attributes, texture),
// runs the rest of the shape list; a query that reaches another mesh goes to the next round's queue,
// a completed query is shaded — material bounce, alpha test, light loop — and either ends the path
// (fold + sample) or begins the next segment, whose shape list runs here as well.
#define RT_SHADE_TILE 1024                   // queue entries a CTA sorts and shades per iteration
template <bool CULL, int MODE>
__global__ void __launch_bounds__(256, RT_SHADE_BLOCKS)
rt_shade_kernel(const DevScene sc, const RenderArgs a, const WaveArgs w, int round)
{
    const unsigned count = w.counts[round] < w.pool.cap ? w.counts[round] : w.pool.cap;
    const unsigned* __restrict__ queue = w.queue[round & 1];
    unsigned* next_queue = w.queue[(round + 1) & 1];
    unsigned* next_count = w.counts + round + 1;
    if (count == 0) return;                     // an empty round (or retry pass) costs a launch, nothing more
    Counters cnt = { 0, 0, 0, 0, 0, 0 };
    // A CTA takes RT_SHADE_TILE consecutive entries at a time and sorts them by the work they need before any of
    // it is done: HEAVY entries (a mesh hit: attributes, texture, material, the next segment's shape list; or a
    // query still in its shape list) first, then LIGHT ones (the walk found nothing and nothing was hit before:
    // usually sky and the fold), entries the walk kernel retired dropped.  Thread t then shades entries t, t + 256,
    // ... of that order, so the lanes of a warp run the same branch (bounce rounds: 1 entry in 4 is heavy — unsorted,
    // 6 of 32 lanes were active in the material code) and every warp gets its share of the heavy ones.  Queue order
    // carries no meaning (a path's RNG, sample slot and stack are its own), so results do not change.
    __shared__ unsigned s_id[RT_SHADE_TILE];
    __shared__ unsigned s_heavy[RT_SHADE_TILE / 32], s_light[RT_SHADE_TILE / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    // (a thin round is spread over as many CTAs as there are: tiles of 256 or 512 entries then)
    const int per_thread = count >= gridDim.x * 1024u ? 4 : (count >= gridDim.x * 512u ? 2 : 1);
    const unsigned tile = 256u * (unsigned)per_thread;
    for (unsigned base = blockIdx.x * tile; base < count; base += gridDim.x * tile)
    {
        unsigned ids[RT_SHADE_TILE / 256];
        int kinds[RT_SHADE_TILE / 256];
        unsigned hms[RT_SHADE_TILE / 256], lms[RT_SHADE_TILE / 256];
#pragma unroll
        for (int j = 0; j < RT_SHADE_TILE / 256; j++)
        {
            const unsigned e = base + (unsigned)j * 256u + threadIdx.x;
            ids[j] = 0; kinds[j] = 2;
            if (j < per_thread && e < count)
            {
                ids[j] = queue[e];
                const int4 cur = w.pool.cur[ids[j]];
                const int st = cur.z & 255;
                if (st != ST_IDLE) kinds[j] = (st == ST_MESHDONE && cur.y < 0 && cur.w == -1) ? 1 : 0;
            }
            hms[j] = __ballot_sync(RT_FULL_MASK, kinds[j] == 0);
            lms[j] = __ballot_sync(RT_FULL_MASK, kinds[j] == 1);
            if (lane == 0) { s_heavy[j * 8 + warp] = (unsigned)__popc(hms[j]); s_light[j * 8 + warp] = (unsigned)__popc(lms[j]); }
        }
        __syncthreads();
        unsigned n_heavy = 0, n_light = 0, heavy_before[RT_SHADE_TILE / 256], light_before[RT_SHADE_TILE / 256];
#pragma unroll
        for (int g = 0; g < RT_SHADE_TILE / 32; g++)
        {
#pragma unroll
            for (int j = 0; j < RT_SHADE_TILE / 256; j++)
                if (g == j * 8 + warp) { heavy_before[j] = n_heavy; light_before[j] = n_light; }
            n_heavy += s_heavy[g]; n_light += s_light[g];
        }
#pragma unroll
        for (int j = 0; j < RT_SHADE_TILE / 256; j++)
        {
            if (kinds[j] == 0) s_id[heavy_before[j] + (unsigned)__popc(hms[j] & lt_mask)] = ids[j];
            else if (kinds[j] == 1) s_id[n_heavy + light_before[j] + (unsigned)__popc(lms[j] & lt_mask)] = ids[j];
        }
        __syncthreads();
        const unsigned n_live = n_heavy + n_light;
        for (unsigned t0 = 0; t0 < n_live; t0 += 256u)
        {
            const unsigned t = t0 + threadIdx.x;
            bool push = false;
            unsigned id = 0;
            if (t < n_live)
            {
                id = s_id[t];
                Query q; PathState s; int state;
                pool_load<MODE>(w.pool, id, q, state, s);
                query_mesh_done(sc, q, state, cnt);
                for (;;)
                {
                    query_shapes<CULL>(sc, q, state, cnt);
                    if (state == ST_TRAVERSE) { push = true; break; }
                    Ray next; next.o = V3(0, 0, 0); next.d = V3(0, 0, 0); next.dist = 0.0f;
                    bool next_any = false;
                    if (!shade_query<MODE>(sc, a, w.pool, id, q, s, next, next_any)) break;
                    query_begin(q, next, next_any, cnt);
                    s.seg_dist = next.dist;
                    state = ST_SHAPES;
                }
                if (push) pool_store<MODE>(w.pool, id, q, state, s);
            }
            // (whole warps get here together: the push wants converged lanes)
            queue_push(next_queue, next_count, push, id);
        }
        __syncthreads();                        // s_id is rewritten by the next tile
    }
    flush_counters(cnt, a.counters, a.exact);
}

// ---- sample fold: AccumulatePixel::AddPixel + GetGammaSpacePixel ---------------------------------------
// (RayTracerProgram.cpp:57-71, :155-185).  One thread per pixel of the task (LIST: per entry of the masked render's
// pixel list; threads past its count idle); streaming.
// MOMENTS (rt_gpu_track_moments): also the Welford update of the pixel's moments per pass colour x, one fp32 rounding per
// operation: with n = Num before the pass, s0 the sum before and s1 = s0 + x after it, M2 += (x - s0 / n) * (x - s1 / (n + 1))
// when n > 0, and .w += 1.
template <bool MOMENTS, bool LIST>
__device__ __forceinline__ void fold_items(const RenderArgs& a, int pass_count)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int pixel;
    if (LIST)
    {
        if ((unsigned)idx >= *a.list_count) return;
        const unsigned item = a.list[idx];
        int x, y;
        pixel = block_pixel(a, item >> 5, (int)(item & 31u), x, y);
    }
    else
    {
        pixel = a.start + idx;
        if (pixel > a.end) return;
        const int x = pixel % a.width, y = pixel / a.width;
        if (!owns_pixel(a, x, y)) return;
    }
    const size_t stride = (size_t)a.width * a.height;
    float4 acc = a.accum[pixel];
    float3 sum = V3(acc.x, acc.y, acc.z);
    int num = (int)acc.w;
    float3 last = V3(0, 0, 0);
    float4 mom = MOMENTS ? a.moments[pixel] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    for (int p = 0; p < pass_count; p++)
    {
        float3 col;
        if (a.antialias)
        {
            const float4 s0 = a.samples[(size_t)(p * 4) * stride + pixel];
            if (s0.w != 0.0f) col = V3(s0.x, s0.y, s0.z);       // the generate kernel folded this pass already (four sky rays)
            else
            {
                col = add3(V3(0, 0, 0), V3(s0.x, s0.y, s0.z));
#pragma unroll
                for (int i = 1; i < 4; i++)
                {
                    const float4 s = a.samples[(size_t)(p * 4 + i) * stride + pixel];
                    col = add3(col, V3(s.x, s.y, s.z));
                }
                col = V3(col.x / 4.0f, col.y / 4.0f, col.z / 4.0f);
            }
        }
        else
        {
            const float4 s = a.samples[(size_t)p * stride + pixel];
            col = V3(s.x, s.y, s.z);
        }
        const float3 before = sum;
        sum = add3(sum, col);
        if (MOMENTS)
        {
            if (num > 0)
            {
                const float n0 = (float)num, n1 = (float)(num + 1);
                mom.x = mom.x + (col.x - before.x / n0) * (col.x - sum.x / n1);
                mom.y = mom.y + (col.y - before.y / n0) * (col.y - sum.y / n1);
                mom.z = mom.z + (col.z - before.z / n0) * (col.z - sum.z / n1);
            }
            mom.w = mom.w + 1.0f;
        }
        num++;
        last = col;
    }
    if (a.mode == RT_MODE_PREVIEW)
    {
        // UseBaseColor: bitcolor only, accuBuffer is left alone (RayTracerProgram.cpp:175-180)
        a.preview[pixel] = make_float4(last.x, last.y, last.z, 1.0f);
        a.display[pixel] = make_pixel(last);
        return;
    }
    a.accum[pixel] = make_float4(sum.x, sum.y, sum.z, (float)num);
    if (MOMENTS) a.moments[pixel] = mom;
    const float fn = (float)num;
    a.display[pixel] = make_pixel(V3(sum.x / fn, sum.y / fn, sum.z / fn));
}

__global__ void rt_resolve_kernel(const RenderArgs a, int pass_count)
{
    fold_items<false, false>(a, pass_count);
}

// the fold of a render that tracks moments (MOMENTS) or renders a pixel list (LIST); <false, false> is rt_resolve_kernel
template <bool MOMENTS, bool LIST>
__global__ void rt_fold_kernel(const RenderArgs a, int pass_count)
{
    fold_items<MOMENTS, LIST>(a, pass_count);
}

__global__ void rt_display_kernel(const float4* accum, uint32_t* display, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 acc = accum[i];
    const int num = (int)acc.w;
    if (num <= 0) { display[i] = 0; return; }
    const float fn = (float)num;
    display[i] = make_pixel(V3(acc.x / fn, acc.y / fn, acc.z / fn));
}
