// rt_bvh_core.hpp — the device BVH builder's core (rt_bvh_build.cu), library-internal: rt_gpu_build_bvh wraps it with
// host copies, rt_gpu_update_mesh (rt_gpu.cu) runs it on device inputs into a mesh's spare arrays.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "rt_gpu.h"

// Device bytes of the scratch block a build of num_tris triangles needs (256-byte aligned base).  Its first 16 bytes
// are the level counters {next segments, largest child, flag, -}; the flag is the caller's (see below).
__attribute__((visibility("hidden"))) size_t rt_bvh_scratch_bytes(int num_tris);
__attribute__((visibility("hidden"))) int* rt_bvh_scratch_flag(void* scratch);

// KdTree::Build of points / indices (DEVICE, indices in range) on `st` into nodes (2T-1) and tris (T), DEVICE.  One
// host read of the level counters per tree level (into `host_counts`, 4 ints, pinned for speed), so the call returns
// once the build is complete on the device.  check_flag: the first read also fetches the scratch flag, which work
// enqueued on `st` before the call has set (the caller zeroes it first); a non-zero flag stops the build with
// RT_ERR_INVALID and `message` as the context's error after the first level (nodes / tris then hold a partial tree).
__attribute__((visibility("hidden"))) int rt_bvh_build_core(rt_gpu_ctx* ctx, const float* points, const int* indices, int num_tris,
                                                            cudaStream_t st, void* scratch, int* host_counts, bool check_flag,
                                                            const char* message, rt_bvh_node* nodes, rt_tri* tris, int* out_depth);
