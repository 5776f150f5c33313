// rt_adaptive.cu — adaptive sampling: per-pixel moments (rt_gpu_track_moments), the mask compaction of
// rt_gpu_render_masked (whose render is rt_gpu.cu's) and the pixel selection from the error estimate (rt_gpu_select_pixels).
#include "rt_context.hpp"

#include <cmath>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

// A work item (block << 5 | lane) of the task `a` that the mask keeps: inside the task (range, tiles, image) and selected
struct MaskedItem
{
    RenderArgs a;
    const uint8_t* mask;
    __device__ __forceinline__ bool operator()(unsigned item) const
    {
        int x, y;
        const int px = block_pixel(a, item >> 5, (int)(item & 31u), x, y);
        return px >= 0 && mask[px] != 0;
    }
};

// The list is in work-item order: 32 consecutive entries come from one 8x4 pixel block or its neighbours, so the camera
// rays of a generate warp stay coherent for the packet walk of round 0.  DeviceSelect keeps the input order, so the list
// (and with it every sample's pool slot and retry item) does not depend on scheduling.
__attribute__((visibility("hidden"))) int compact_mask(rt_gpu_ctx* ctx, const RenderArgs& a, const uint8_t* mask,
                                                       const unsigned** list, const unsigned** count)
{
    const unsigned n = a.num_blocks * 32u;          // below 2^32: render() checks one pass's work list
    const MaskedItem keep = { a, mask };
    const thrust::counting_iterator<unsigned> items(0u);
    size_t temp = 0;
    RT_CUDA(cub::DeviceSelect::If(nullptr, temp, items, (unsigned*)nullptr, (unsigned*)nullptr, n, keep, ctx->stream));
    // scratch: [count | list of n | CUB's temporaries], 256-byte aligned parts
    const size_t list_at = 256, temp_at = (list_at + (size_t)n * sizeof(unsigned) + 255) & ~(size_t)255;
    SlotAdaptive& s = ctx->adapt;
    if (temp_at + temp > s.scratch_cap)
    {
        // stream-ordered: the slot's earlier calls (joined back into its stream) are done with the old block first
        if (s.scratch) RT_CUDA(cudaFreeAsync(s.scratch, ctx->stream));
        s.scratch = nullptr; s.scratch_cap = 0;
        RT_CUDA(cudaMallocAsync(&s.scratch, temp_at + temp, ctx->stream));
        s.scratch_cap = temp_at + temp;
    }
    char* base = (char*)s.scratch;
    RT_CUDA(cub::DeviceSelect::If(base + temp_at, temp, items, (unsigned*)(base + list_at), (unsigned*)base, n, keep, ctx->stream));
    ctx->launches += 2;                             // the tile-state initialisation and the selection sweep
    *list = (const unsigned*)(base + list_at);
    *count = (const unsigned*)base;
    return RT_OK;
}

// One thread per pixel of the frame: mask = 1 iff the pixel is in the region, Num < max_passes and (Num < min_passes, or
// the moments do not cover every pass, or some channel's standard error exceeds abs_tol + rel_tol * luminance).
__global__ void rt_select_pixels_kernel(const float4* __restrict__ accum, const float4* __restrict__ moments, const RenderArgs a,
                                        rt_select_params s, uint8_t* __restrict__ mask, int* __restrict__ count)
{
    const int npix = a.width * a.height;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool sel = false;
    if (i < npix && i >= a.start && i <= a.end && owns_pixel(a, i % a.width, i / a.width))
    {
        const float4 acc = accum[i];
        const int n = (int)acc.w;
        if (n < s.max_passes)
        {
            const float4 m = moments[i];
            if (n < s.min_passes || m.w != (float)n) sel = true;
            else
            {
                const float fn = (float)n, fn1 = (float)(n - 1);
                const float se_r = sqrtf((m.x / fn1) / fn), se_g = sqrtf((m.y / fn1) / fn), se_b = sqrtf((m.z / fn1) / fn);
                const float lum = (0.2126f * (acc.x / fn) + 0.7152f * (acc.y / fn)) + 0.0722f * (acc.z / fn);
                const float tol = s.abs_tol + s.rel_tol * lum;
                sel = se_r > tol || se_g > tol || se_b > tol;       // NaN compares false: it selects nothing
            }
        }
    }
    if (i < npix) mask[i] = sel ? 1 : 0;
    const unsigned votes = __ballot_sync(RT_FULL_MASK, sel);
    if ((threadIdx.x & 31) == 0 && votes) atomicAdd(count, __popc(votes));
}

extern "C" {

int rt_gpu_track_moments(rt_gpu_ctx* ctx, int32_t on)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!on) { ctx->adapt.track = false; return RT_OK; }
        RT_CUDA(cudaSetDevice(ctx->device));
        const size_t n = (size_t)ctx->width * ctx->height;
        if (n > 0)
        {
            if (!ctx->adapt.moments) RT_CUDA(cudaMalloc((void**)&ctx->adapt.moments, n * sizeof(float4)));
            RT_CUDA(cudaMemsetAsync(ctx->adapt.moments, 0, n * sizeof(float4), ctx->stream));
        }
        ctx->adapt.track = true;                    // (no frame yet: rt_gpu_reset_accum allocates the buffer with the frame)
        return RT_OK;
    });
}

int rt_gpu_select_pixels(rt_gpu_ctx* ctx, const rt_render_params* region, const rt_select_params* s, uint8_t* mask,
                         int32_t* count, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!region || !s) return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: region and select params are required");
        if (s->min_passes < 2 || s->max_passes < s->min_passes)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: need 2 <= min_passes <= max_passes");
        if (!std::isfinite(s->abs_tol) || !std::isfinite(s->rel_tol) || s->abs_tol < 0.0f || s->rel_tol < 0.0f)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: tolerances must be finite and >= 0");
        if (!ctx->adapt.moments)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: moments have not been tracked on this frame slot (rt_gpu_track_moments)");
        if (region->width != ctx->width || region->height != ctx->height)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: region size differs from the frame slot's frame");
        const int npix = ctx->width * ctx->height;
        if (region->start < 0 || region->end >= npix) return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: pixel range outside the frame");
        if (region->tile_count > 1 && (region->tile_size <= 0 || region->tile_rank < 0 || region->tile_rank >= region->tile_count))
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: bad tile ownership fields");
        if (!mask || !count) return fail(ctx, RT_ERR_INVALID, "rt_gpu_select_pixels: mask and count are required");
        int rc = check_device_args(ctx, "rt_gpu_select_pixels", { { mask, "mask", 1 }, { count, "count", 4 } });
        if (rc != RT_OK) return rc;
        RT_CUDA(cudaSetDevice(ctx->device));
        RenderArgs a;
        memset(&a, 0, sizeof a);
        a.width = region->width; a.height = region->height; a.start = region->start; a.end = region->end;
        a.tiled = region->tile_count > 1 ? 1 : 0;
        a.tile_size = region->tile_size; a.tile_count = region->tile_count; a.tile_rank = region->tile_rank;
        if (a.tiled) a.tiles_x = (region->width + region->tile_size - 1) / region->tile_size;
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RT_CUDA(order_streams(ctx, st, ctx->stream));
        RT_CUDA(cudaMemsetAsync(count, 0, sizeof(int32_t), ctx->stream));
        rt_select_pixels_kernel<<<(npix + 255) / 256, 256, 0, ctx->stream>>>(ctx->accum, ctx->adapt.moments, a, *s, mask, count);
        RT_CUDA(cudaGetLastError());
        ctx->launches++;
        RT_CUDA(order_streams(ctx, ctx->stream, st));
        return RT_OK;
    });
}

}   // extern "C"
