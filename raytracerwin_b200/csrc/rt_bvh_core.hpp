// rt_bvh_core.hpp — the device BVH builder's core (rt_bvh_build.cu), library-internal: rt_gpu_build_bvh wraps it with
// host copies, rt_gpu_update_mesh and rt_gpu_replace_mesh (rt_scene_edit.cu) run it on device inputs into a mesh's spare
// arrays.  Carve lays out the builder's scratch block and the scene edits' scratch.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stddef.h>

#include "rt_gpu.h"

// Arrays cut one after another from a block whose base is 256-byte aligned, each 256-byte aligned.  On a null base the
// pointers are meaningless and `off` ends as the block's size.
struct Carve
{
    char* base; size_t off;
    template <typename T> T* take(size_t n)
    {
        T* p = (T*)(base + off);
        off += ((n ? n : 1) * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
};

// Device bytes of the scratch block a build of num_tris triangles needs (256-byte aligned base).  Its first 16 bytes
// are the level counters {next segments, largest child, flag, -}; the flag is the caller's: the builder leaves it alone.
__attribute__((visibility("hidden"))) size_t rt_bvh_scratch_bytes(int num_tris);
__attribute__((visibility("hidden"))) int* rt_bvh_scratch_flag(void* scratch);

// KdTree::Build of points / indices (DEVICE, indices in range) on `st` into nodes (2T-1) and tris (T), DEVICE.  One
// host read of the level counters per tree level (into `host_counts`, 4 ints, pinned for speed), so the call returns
// once the build is complete on the device.  The points must be finite (the callers refuse others before the build).
__attribute__((visibility("hidden"))) int rt_bvh_build_core(rt_gpu_ctx* ctx, const float* points, const int* indices, int num_tris,
                                                            cudaStream_t st, void* scratch, int* host_counts, rt_bvh_node* nodes,
                                                            rt_tri* tris, int* out_depth);

// v, with a NaN in the bits the host layer's arithmetic gives it.  Finite corners whose edge products overflow make a
// face normal NaN (inf - inf, inf * 0): x86 writes its default NaN 0xFFC00000 and carries it through every later
// operation, the device writes 0x7FFFFFFF.  Records written on the device take the host's bits, so that a mesh built or
// edited here is byte for byte the host build of the same geometry.
static __device__ __forceinline__ float rt_host_nan(float v) { return v != v ? __uint_as_float(0xFFC00000u) : v; }

// The leaf record of triangle t with corners p0, p1, p2, as the host builder emits it: pads 0 and the face normal
// exactly as RRay.cpp:138-145 computes it (cross(p1-p0, p2-p0), normalised unless |n|^2 < FLT_EPSILON).  The builder's
// k_nodes and rt_gpu_refit_mesh both write it.
static __device__ __forceinline__ rt_tri rt_tri_record(const float* p0, const float* p1, const float* p2, int t)
{
    rt_tri r;
    r.p0[0] = p0[0]; r.p0[1] = p0[1]; r.p0[2] = p0[2]; r.index = t;
    r.p1[0] = p1[0]; r.p1[1] = p1[1]; r.p1[2] = p1[2]; r.pad0 = 0.0f;
    r.p2[0] = p2[0]; r.p2[1] = p2[1]; r.p2[2] = p2[2]; r.pad1 = 0.0f;
    const float ax = p1[0] - p0[0], ay = p1[1] - p0[1], az = p1[2] - p0[2];
    const float bx = p2[0] - p0[0], by = p2[1] - p0[1], bz = p2[2] - p0[2];
    float nx = ay * bz - az * by, ny = az * bx - ax * bz, nz = ax * by - ay * bx;
    const float sqr = nx * nx + ny * ny + nz * nz;
    if (!(fabsf(sqr) < FLT_EPSILON))
    {
        const float inv = 1.0f / sqrtf(sqr);
        nx *= inv; ny *= inv; nz *= inv;
    }
    r.n[0] = rt_host_nan(nx); r.n[1] = rt_host_nan(ny); r.n[2] = rt_host_nan(nz); r.pad2 = 0.0f;
    return r;
}
