// rt_denoise.cu — the guided a-trous denoiser (rt_gpu_denoise): the filter of include/rt_gpu.h on the current frame
// slot's mean colour, guided by the slot's RT_MODE_GUIDES render (shape id, distance, normal) and its moments.
// Compiled with -fmad=false and IEEE div/sqrt, like every device file: each operation below rounds once, in the order
// written, which is what the header states and tests/test_denoise.py restates.
#include "rt_context.hpp"

#include <cmath>

#define RT_DN_BX 16
#define RT_DN_BY 8
#define RT_DN_INVALID (-2)          // the shape id of an invalid pixel: never equal to a valid pixel's (>= -1)

// The per-pixel records the levels read: {x.rgb, v} (ping-pong, one buffer per level parity), {N.xyz, z} and the shape id
// (RT_DN_INVALID for a pixel the filter passes through).  Level 0 writes all three.
struct DenoiseBufs
{
    float4* xv[2];
    float4* nz;
    int* shape;
};

__device__ __forceinline__ float dn_lum(float r, float g, float b) { return (0.2126f * r + 0.7152f * g) + 0.0722f * b; }

__device__ __forceinline__ bool dn_finite3(float4 v) { return isfinite(v.x) && isfinite(v.y) && isfinite(v.z); }

// d = the albedo the pixel's colour is divided by (1 without use_albedo)
__device__ __forceinline__ float3 dn_albedo(const float4* __restrict__ preview, int i)
{
    if (!preview) return make_float3(1.0f, 1.0f, 1.0f);
    const float4 a = preview[i];
    return make_float3(a.x > 1e-3f ? a.x : 1e-3f, a.y > 1e-3f ? a.y : 1e-3f, a.z > 1e-3f ? a.z : 1e-3f);
}

// Level 0: the signal x, its variance v and the guides of every pixel (preview / moments: null when not used)
__global__ void rt_denoise_prep_kernel(const float4* __restrict__ accum, const float4* __restrict__ preview,
                                       const float4* __restrict__ moments, const int2* __restrict__ prim_ids,
                                       const float* __restrict__ prim_dist, const float4* __restrict__ guide, int width,
                                       int height, DenoiseBufs b)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= width || y >= height) return;
    const int i = y * width + x;
    const float4 acc = accum[i];
    const int n = (int)acc.w;
    const bool valid = n > 0 && dn_finite3(acc);
    float4 xv = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (valid)
    {
        const float fn = (float)n;
        const float3 d = dn_albedo(preview, i);
        xv.x = (acc.x / fn) / d.x; xv.y = (acc.y / fn) / d.y; xv.z = (acc.z / fn) / d.z;
        if (moments && n >= 2)
        {
            const float4 m = moments[i];
            if (m.w == fn)
            {
                float v = (dn_lum(m.x, m.y, m.z) / (float)(n - 1)) / fn;
                if (preview)
                {
                    const float yd = dn_lum(d.x, d.y, d.z);
                    v = v / (yd * yd);
                }
                xv.w = v;
            }
        }
    }
    const float4 g = guide[i];
    b.xv[0][i] = xv;
    b.nz[i] = make_float4(g.x, g.y, g.z, prim_dist[i]);
    b.shape[i] = valid ? prim_ids[i].x : RT_DN_INVALID;
}

// Level `step` = 2^k: {x, v} from `in` to `out`.  LAST: the output rules instead, into rgba / argb.
template <bool LAST>
__global__ void __launch_bounds__(RT_DN_BX * RT_DN_BY)
rt_denoise_level_kernel(const float4* __restrict__ in, float4* __restrict__ out, const float4* __restrict__ nz,
                        const int* __restrict__ shape, int width, int height, int step, rt_denoise_params p,
                        const float4* __restrict__ accum, const float4* __restrict__ preview, float4* __restrict__ rgba,
                        uint32_t* __restrict__ argb)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= width || y >= height) return;
    const int i = y * width + x;
    const int sp = shape[i];
    float4 xv = in[i];
    if (sp != RT_DN_INVALID)
    {
        const float H[5] = { 0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f };
        const float4 gp = nz[i];
        const bool hit = sp >= 0;
        const float yp = dn_lum(xv.x, xv.y, xv.z);
        const float lum_scale = p.sigma_lum * sqrtf(xv.w) + p.lum_floor;
        const float depth_scale = (p.sigma_depth * (float)step) * gp.w;
        float W = 0.0f, V = 0.0f, X0 = 0.0f, X1 = 0.0f, X2 = 0.0f;
#pragma unroll
        for (int j = -2; j <= 2; j++)
        {
            const int qy = y + step * j;
            if (qy < 0 || qy >= height) continue;
#pragma unroll
            for (int ii = -2; ii <= 2; ii++)
            {
                const int qx = x + step * ii;
                if (qx < 0 || qx >= width) continue;
                const int q = qy * width + qx;
                float w;
                float4 xq;
                if (ii == 0 && j == 0) { w = 0.140625f; xq = xv; }
                else
                {
                    if (shape[q] != sp) continue;           // also every invalid tap
                    xq = in[q];
                    w = H[ii + 2] * H[j + 2];
                    if (hit)
                    {
                        const float4 gq = nz[q];
                        float wn = (gp.x * gq.x + gp.y * gq.y) + gp.z * gq.z;
                        wn = wn > 0.0f ? wn : 0.0f;
                        for (int k = 0; k < p.normal_log2; k++) wn = wn * wn;
                        const float wz = 1.0f / (1.0f + fabsf(gp.w - gq.w) / depth_scale);
                        w = (w * wn) * wz;
                    }
                    const float t = fabsf(yp - dn_lum(xq.x, xq.y, xq.z)) / lum_scale;
                    w = w * (1.0f / (1.0f + t * t));
                    if (!isfinite(w)) continue;
                }
                W = W + w;
                X0 = X0 + w * xq.x; X1 = X1 + w * xq.y; X2 = X2 + w * xq.z;
                V = V + (w * w) * xq.w;
            }
        }
        xv = make_float4(X0 / W, X1 / W, X2 / W, V / (W * W));
    }
    if (!LAST) { out[i] = xv; return; }
    const float4 acc = accum[i];
    const int n = (int)acc.w;
    float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (n > 0)
    {
        const float fn = (float)n;
        if (!dn_finite3(acc)) o = make_float4(acc.x / fn, acc.y / fn, acc.z / fn, fn);
        else
        {
            const float3 d = dn_albedo(preview, i);
            o = make_float4(xv.x * d.x, xv.y * d.y, xv.z * d.z, fn);
        }
    }
    rgba[i] = o;
    if (argb) argb[i] = n > 0 ? make_pixel(V3(o.x, o.y, o.z)) : 0u;
}

extern "C" {

int rt_gpu_denoise(rt_gpu_ctx* ctx, const rt_denoise_params* p, float* rgba, uint32_t* argb, void* stream)
{
    return rt_guard(ctx, [&]() -> int {
        if (!ctx) return RT_ERR_INVALID;
        if (!p) return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: params are required");
        if (p->levels < 1 || p->levels > 6) return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: levels must be in [1, 6]");
        if ((p->use_albedo != 0 && p->use_albedo != 1) || (p->use_variance != 0 && p->use_variance != 1))
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: use_albedo and use_variance must be 0 or 1");
        if (p->normal_log2 < 0 || p->normal_log2 > 8) return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: normal_log2 must be in [0, 8]");
        if (!std::isfinite(p->sigma_lum) || !std::isfinite(p->sigma_depth) || !std::isfinite(p->lum_floor) ||
            !(p->sigma_lum >= 0.0f) || !(p->sigma_depth > 0.0f) || !(p->lum_floor > 0.0f))
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: need finite sigma_lum >= 0, sigma_depth > 0 and lum_floor > 0");
        if (!ctx->accum || ctx->width <= 0 || ctx->height <= 0) return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: the frame slot has no frame");
        if (!ctx->den.guides || !ctx->den.guide)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: no RT_MODE_GUIDES render on this frame slot since its frame was allocated");
        if (p->use_albedo && !ctx->preview)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: use_albedo without an RT_MODE_PREVIEW pass on this frame slot");
        if (p->use_variance && !ctx->adapt.moments)
            return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: use_variance, but moments have never been tracked on this frame slot");
        if (!rgba) return fail(ctx, RT_ERR_INVALID, "rt_gpu_denoise: rgba is required");
        const int rc = check_device_args(ctx, "rt_gpu_denoise", { { rgba, "rgba", 16 }, { argb, "argb", 4 } });
        if (rc != RT_OK) return rc;
        RT_CUDA(cudaSetDevice(ctx->device));
        const int width = ctx->width, height = ctx->height;
        const size_t npix = (size_t)width * height;
        // scratch: [xv ping | xv pong | nz | shape], 256-byte aligned parts
        const size_t f4 = (npix * sizeof(float4) + 255) & ~(size_t)255;
        const size_t need = 3 * f4 + ((npix * sizeof(int) + 255) & ~(size_t)255);
        const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RT_CUDA(order_streams(ctx, st, ctx->stream));
        SlotDenoise& s = ctx->den;
        if (need > s.scratch_cap)
        {
            // stream-ordered: the slot's earlier denoise calls are done with the old block first
            if (s.scratch) RT_CUDA(cudaFreeAsync(s.scratch, ctx->stream));
            s.scratch = nullptr; s.scratch_cap = 0;
            RT_CUDA(cudaMallocAsync(&s.scratch, need, ctx->stream));
            s.scratch_cap = need;
        }
        char* base = (char*)s.scratch;
        DenoiseBufs b;
        b.xv[0] = (float4*)base; b.xv[1] = (float4*)(base + f4); b.nz = (float4*)(base + 2 * f4); b.shape = (int*)(base + 3 * f4);
        const float4* preview = p->use_albedo ? ctx->preview : nullptr;
        const dim3 block(RT_DN_BX, RT_DN_BY), grid((width + RT_DN_BX - 1) / RT_DN_BX, (height + RT_DN_BY - 1) / RT_DN_BY);
        rt_denoise_prep_kernel<<<grid, block, 0, ctx->stream>>>(ctx->accum, preview, p->use_variance ? ctx->adapt.moments : nullptr,
                                                                ctx->prim_ids, ctx->prim_dist, ctx->den.guide, width, height, b);
        RT_CUDA(cudaGetLastError());
        ctx->launches++;
        for (int k = 0; k < p->levels; k++)
        {
            const float4* in = b.xv[k & 1];
            float4* out = b.xv[(k + 1) & 1];
            if (k + 1 < p->levels)
                rt_denoise_level_kernel<false><<<grid, block, 0, ctx->stream>>>(in, out, b.nz, b.shape, width, height, 1 << k, *p,
                                                                                nullptr, nullptr, nullptr, nullptr);
            else
                rt_denoise_level_kernel<true><<<grid, block, 0, ctx->stream>>>(in, nullptr, b.nz, b.shape, width, height, 1 << k, *p,
                                                                               ctx->accum, preview, (float4*)rgba, argb);
            RT_CUDA(cudaGetLastError());
            ctx->launches++;
        }
        RT_CUDA(order_streams(ctx, ctx->stream, st));
        return RT_OK;
    });
}

}   // extern "C"
