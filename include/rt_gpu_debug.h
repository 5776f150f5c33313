/* rt_gpu_debug.h — tooling entry points of librt_b200.so (tools/render_once.py, tools/timeline.py).
 *
 * Not part of the drop-in boundary (include/rt_gpu.h): nothing here replaces a reference interface.  They read
 * the per-round bookkeeping of the wavefront after a render call made with rt_gpu_time_kernels(ctx, 1), so that
 * the round structure can be inspected without a profiler; rt_gpu_debug_read_mesh reads a mesh's device arrays back.
 * Every function synchronises the context. */
#ifndef RT_GPU_DEBUG_H
#define RT_GPU_DEBUG_H

#include "rt_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Entries of each round of the last batch on pipe 0 (counts[k], k < max_rounds) and the walk-kernel time of
 * each timed bracket (ms[k]); counts[max_rounds - 1] is overwritten with the longest single walk (node steps).
 * Returns the number of timed brackets, or a negative rt_status. */
int rt_gpu_debug_rounds(rt_gpu_ctx* ctx, uint32_t* counts, float* ms, int32_t max_rounds);

/* Begin / end of every timed walk bracket of the last call in ms since the call began (launch order: chunk by
 * chunk, round by round).  Returns the number of brackets written (<= cap), or a negative rt_status. */
int rt_gpu_debug_timeline(rt_gpu_ctx* ctx, float* begin_ms, float* end_ms, int32_t cap);

/* Long-walk queue sizes per round of the last batch on pipe 0. */
int rt_gpu_debug_long(rt_gpu_ctx* ctx, uint32_t* lcounts, int32_t max_rounds);

/* The current device arrays of mesh `mesh` (after every update enqueued so far): nodes (the uploaded num_nodes records,
 * 2 * num_tris - 1 for a tree of its triangles and after any update; inner nodes
 * with the right child in `tri` as the device keeps them), tris and shade (num_tris each, shade in LEAF order), the
 * bounds {min xyz, max xyz} of the shape that references it and its culling margin.  Any output may be NULL. */
int rt_gpu_debug_read_mesh(rt_gpu_ctx* ctx, int32_t mesh, rt_bvh_node* nodes, rt_tri* tris, rt_shade* shade, float* bounds6,
                           float* cull_scale);

/* The material and light records the kernels read now (after every update enqueued so far): the first min(count, cap)
 * of each (either array may be NULL), and counts2 = {material count, light count}. */
int rt_gpu_debug_read_appearance(rt_gpu_ctx* ctx, rt_material* materials, int32_t mat_cap, rt_light* lights, int32_t light_cap,
                                 int32_t* counts2);

/* The texels of texture `slot` of mesh `mesh` as the atlas holds them now: height x width x {r,g,b,a} floats (the slot's
 * uploaded size). */
int rt_gpu_debug_read_texture(rt_gpu_ctx* ctx, int32_t mesh, int32_t slot, float* rgba);

#ifdef __cplusplus
}
#endif
#endif
