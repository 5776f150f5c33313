// rt_bvh_build.cu — the reference's "KdTree" build (KdNode::Build, KdTree.cpp:10-126) on the GPU, emitting the
// same pre-order, escape-threaded arrays as the host builder (host/bvh_build.cpp) BIT FOR BIT.
//
// SURVEY.md §8(f) rank 1.  The tree shape decides traversal order and therefore which of two near-equal hits
// wins, so every rule is the reference's:
//   node bounds   min/max over the corners of the node's triangles, strict </> in list order: the FIRST corner
//                 that attains the extreme supplies the bits (matters for -0 vs +0)            (KdTree.cpp:42-47)
//   split axis    widest extent, x only if strictly wider than y and z, y only if strictly wider than z (:10-35)
//   split value   mean of the triangle centroids (v0+v1+v2)/3, SUMMED IN LIST ORDER in fp32   (:57-66)
//   partition     centroid[axis] < mean goes left, list order kept (stable)                    (:72-105)
//   fallback      all on one side -> first half / second half                                  (:108-113)
// Level-synchronous: every tree level is a handful of launches over all triangle positions.  Everything is
// order-independent or an exact integer scan, except the fp32 centroid sum, which is not associative: it is
// accumulated sequentially per node — one FADD chain per component, fed from shared-memory tiles that a second
// warp streams in (k_sum_big) — the only serial part (~4 cycles per triangle of the largest node of a level).
// Pre-order indices need no second pass: a node with c triangles owns 2c-1 nodes, so left child = node+1,
// right child = node + 2*count_left, escape = node + 2c-1, and leaf k of the final order is triangle slot k.
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "rt_gpu.h"
#include "rt_bvh_core.hpp"

// library-internal helpers of rt_gpu.cu (the context is opaque here too)
__attribute__((visibility("hidden"))) int rt_ctx_device(rt_gpu_ctx* ctx);
__attribute__((visibility("hidden"))) void rt_ctx_set_error(rt_gpu_ctx* ctx, const char* msg);

namespace {

struct Seg { int begin, end, node; };

struct Level
{
    const float* P; const int* I;
    const float* cx; const float* cy; const float* cz;      // centroids by triangle id
    float* gx; float* gy; float* gz;                         // centroids by position (gathered every level)
    int* order; int* order_next;
    int* seg_of_pos; int* seg_of_pos_next;
    const Seg* segs; Seg* segs_next;
    int num_segs; int* next_count;
    unsigned long long* kmin; unsigned long long* kmax;     // [num_segs * 3]
    float* mean; int* axis; int* nl;                         // per segment
    float* big_sum; int* max_count;                          // serial sums of the big segments; largest child of the level
    int* flags; int* pre;                                    // per position (+1)
    rt_bvh_node* nodes; rt_tri* tris;
    int T;
};

__device__ __forceinline__ unsigned ord_bits(float v)
{
    unsigned b = __float_as_uint(v);
    if (v == 0.0f) b = 0u;                                   // -0 and +0 compare equal in the reference
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void k_centroids(const float* P, const int* I, int T, float* cx, float* cy, float* cz, int* order, int* seg_of_pos)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const float* v0 = P + 3 * (size_t)I[3 * t], * v1 = P + 3 * (size_t)I[3 * t + 1], * v2 = P + 3 * (size_t)I[3 * t + 2];
    // (v0 + v1 + v2) / 3.0f, component-wise, left to right (KdTree.cpp:60-63)
    cx[t] = ((v0[0] + v1[0]) + v2[0]) / 3.0f;
    cy[t] = ((v0[1] + v1[1]) + v2[1]) / 3.0f;
    cz[t] = ((v0[2] + v1[2]) + v2[2]) / 3.0f;
    order[t] = t;
    seg_of_pos[t] = 0;
}

__global__ void k_init_keys(unsigned long long* kmin, unsigned long long* kmax, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { kmin[i] = ~0ull; kmax[i] = 0ull; }
}

// per position: the six extreme keys of its triangle, merged into its segment's keys
__global__ void k_bounds(Level L)
{
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int seg = -1;
    unsigned long long mn[3] = { ~0ull, ~0ull, ~0ull }, mx[3] = { 0ull, 0ull, 0ull };
    if (pos < L.T)
    {
        seg = L.seg_of_pos[pos];
        if (seg >= 0)
        {
            const int t = L.order[pos];
            for (int k = 0; k < 3; k++)
            {
                const float* p = L.P + 3 * (size_t)L.I[3 * t + k];
                const unsigned sub = (unsigned)pos * 3u + (unsigned)k;
                for (int c = 0; c < 3; c++)
                {
                    const float v = p[c];
                    if (v != v) continue;                                   // NaN never wins a < or > test
                    const unsigned long long o = (unsigned long long)ord_bits(v) << 32;
                    const unsigned long long a = o | sub, b = o | (0xFFFFFFFFu - sub);
                    if (a < mn[c]) mn[c] = a;
                    if (b > mx[c]) mx[c] = b;
                }
            }
        }
    }
    // warp-aggregate when the whole warp sits in one segment (the usual case for all but the tiniest nodes)
    const int seg0 = __shfl_sync(0xffffffffu, seg, 0);
    if (__all_sync(0xffffffffu, seg == seg0))
    {
        if (seg0 < 0) return;
        for (int c = 0; c < 3; c++)
            for (int o = 16; o > 0; o >>= 1)
            {
                const unsigned long long a = __shfl_xor_sync(0xffffffffu, mn[c], o), b = __shfl_xor_sync(0xffffffffu, mx[c], o);
                if (a < mn[c]) mn[c] = a;
                if (b > mx[c]) mx[c] = b;
            }
        if (lane == 0)
            for (int c = 0; c < 3; c++)
            {
                atomicMin(L.kmin + 3 * (size_t)seg0 + c, mn[c]);
                atomicMax(L.kmax + 3 * (size_t)seg0 + c, mx[c]);
            }
    }
    else if (seg >= 0)
        for (int c = 0; c < 3; c++)
        {
            atomicMin(L.kmin + 3 * (size_t)seg + c, mn[c]);
            atomicMax(L.kmax + 3 * (size_t)seg + c, mx[c]);
        }
}

__device__ __forceinline__ float key_value(const Level& L, unsigned long long key, bool is_max, int c, float none)
{
    if (is_max ? key == 0ull : key == ~0ull) return none;
    const unsigned low = (unsigned)(key & 0xFFFFFFFFull);
    const unsigned sub = is_max ? 0xFFFFFFFFu - low : low;
    const int pos = (int)(sub / 3u), k = (int)(sub % 3u);
    const int t = L.order[pos];
    return L.P[3 * (size_t)L.I[3 * t + k] + c];
}

// centroids in list order, so that the serial sum below streams through contiguous memory
__global__ void k_gather(Level L)
{
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= L.T) return;
    if (L.seg_of_pos[pos] < 0) return;
    const int t = L.order[pos];
    L.gx[pos] = L.cx[t]; L.gy[pos] = L.cy[t]; L.gz[pos] = L.cz[t];
}

// The serial centroid sum of a BIG segment (KdTree.cpp:57-66): 4 cycles per triangle on one FADD chain per
// component is the floor, so the point is to keep that chain fed.  One 64-thread block per segment: warp 1
// streams tiles of the gathered centroids into shared memory (coalesced), lane 0 of warp 0 adds the previous
// tile in list order meanwhile (double buffer, one __syncthreads per tile).
#define BIG_SEG 512
#define SUM_TILE 1024
__global__ void __launch_bounds__(64) k_sum_big(Level L)
{
    __shared__ float tile[2][3][SUM_TILE];
    const int s = blockIdx.x;
    const Seg sg = L.segs[s];
    const int count = sg.end - sg.begin;
    if (count <= BIG_SEG) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntiles = (count + SUM_TILE - 1) / SUM_TILE;
    float sx = 0.0f, sy = 0.0f, sz = 0.0f;
    for (int k = 0; k <= ntiles; k++)
    {
        if (warp == 1 && k < ntiles)
        {
            const int base = sg.begin + k * SUM_TILE;
            const int n = sg.end - base < SUM_TILE ? sg.end - base : SUM_TILE;
            float* tx = tile[k & 1][0]; float* ty = tile[k & 1][1]; float* tz = tile[k & 1][2];
            for (int j = lane; j < n; j += 32) { tx[j] = L.gx[base + j]; ty[j] = L.gy[base + j]; tz[j] = L.gz[base + j]; }
        }
        if (warp == 0 && lane == 0 && k > 0)
        {
            const int base = sg.begin + (k - 1) * SUM_TILE;
            const int n = sg.end - base < SUM_TILE ? sg.end - base : SUM_TILE;
            const float* tx = tile[(k - 1) & 1][0]; const float* ty = tile[(k - 1) & 1][1]; const float* tz = tile[(k - 1) & 1][2];
            int j = 0;
            for (; j + 8 <= n; j += 8)
            {
#pragma unroll
                for (int u = 0; u < 8; u++) { sx += tx[j + u]; sy += ty[j + u]; sz += tz[j + u]; }
            }
            for (; j < n; j++) { sx += tx[j]; sy += ty[j]; sz += tz[j]; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { L.big_sum[3 * (size_t)s] = sx; L.big_sum[3 * (size_t)s + 1] = sy; L.big_sum[3 * (size_t)s + 2] = sz; }
}

// One THREAD per segment: bounds from the keys, the sequential centroid sum, mean, axis; node record; leaf record.
__global__ void k_nodes(Level L)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= L.num_segs) return;
    const Seg sg = L.segs[s];
    const int count = sg.end - sg.begin;
    float mn[3], mx[3];
    for (int c = 0; c < 3; c++)
    {
        mn[c] = key_value(L, L.kmin[3 * (size_t)s + c], false, c, FLT_MAX);
        mx[c] = key_value(L, L.kmax[3 * (size_t)s + c], true, c, -FLT_MAX);
    }
    rt_bvh_node nd;
    nd.bmin[0] = mn[0]; nd.bmin[1] = mn[1]; nd.bmin[2] = mn[2];
    nd.bmax[0] = mx[0]; nd.bmax[1] = mx[1]; nd.bmax[2] = mx[2];
    nd.escape = sg.node + 2 * count - 1;
    nd.tri = count == 1 ? sg.begin : -1;
    L.nodes[sg.node] = nd;
    if (count == 1)
    {
        const int t = L.order[sg.begin];
        const float* p0 = L.P + 3 * (size_t)L.I[3 * t], * p1 = L.P + 3 * (size_t)L.I[3 * t + 1], * p2 = L.P + 3 * (size_t)L.I[3 * t + 2];
        L.tris[sg.begin] = rt_tri_record(p0, p1, p2, t);
        L.axis[s] = -1;
        return;
    }
    // fp32 sum in list order (KdTree.cpp:57-66): one serial chain per component; the loads run ahead of it
    float sx = 0.0f, sy = 0.0f, sz = 0.0f;
    if (count > BIG_SEG) { sx = L.big_sum[3 * (size_t)s]; sy = L.big_sum[3 * (size_t)s + 1]; sz = L.big_sum[3 * (size_t)s + 2]; }
    else for (int i = sg.begin; i < sg.end; i++) { sx += L.gx[i]; sy += L.gy[i]; sz += L.gz[i]; }
    const float fc = (float)count;
    const float ex = mx[0] - mn[0], ey = mx[1] - mn[1], ez = mx[2] - mn[2];
    int axis;
    if (ex > ey) axis = (ex > ez) ? 0 : 2;
    else axis = (ey > ez) ? 1 : 2;
    L.axis[s] = axis;
    L.mean[s] = (axis == 0 ? sx : (axis == 1 ? sy : sz)) / fc;
}

__global__ void k_flags(Level L)
{
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= L.T) return;
    const int seg = L.seg_of_pos[pos];
    int f = 0;
    if (seg >= 0)
    {
        const int axis = L.axis[seg];
        if (axis >= 0)
        {
            const int t = L.order[pos];
            const float v = axis == 0 ? L.cx[t] : (axis == 1 ? L.cy[t] : L.cz[t]);
            f = v < L.mean[seg] ? 1 : 0;
        }
    }
    L.flags[pos] = f;
}

// exclusive scan of `in[0..n)` into `out[0..n]` (out[n] = total): block sums, scan of sums, block scans
#define SCAN_BLOCK 1024
__global__ void k_block_sums(const int* in, int n, int* sums)
{
    __shared__ int sh[32];
    const int i = blockIdx.x * SCAN_BLOCK + threadIdx.x;
    int v = i < n ? in[i] : 0;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32)
    {
        int w = sh[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
        if (threadIdx.x == 0) sums[blockIdx.x] = w;
    }
}

__global__ void k_scan_sums(int* sums, int nb)          // one block; exclusive, in place; sums[nb] = total
{
    __shared__ int sh[SCAN_BLOCK];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nb; base += SCAN_BLOCK)
    {
        const int i = base + threadIdx.x;
        const int v = i < nb ? sums[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < SCAN_BLOCK; o <<= 1)
        {
            const int a = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += a;
            __syncthreads();
        }
        const int incl = sh[threadIdx.x];
        if (i < nb) sums[i] = carry + incl - v;
        __syncthreads();
        if (threadIdx.x == SCAN_BLOCK - 1) carry += incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[nb] = carry;
}

__global__ void k_block_scan(const int* in, int n, const int* sums, int* out)
{
    __shared__ int sh[SCAN_BLOCK];
    const int i = blockIdx.x * SCAN_BLOCK + threadIdx.x;
    const int v = i < n ? in[i] : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < SCAN_BLOCK; o <<= 1)
    {
        const int a = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += a;
        __syncthreads();
    }
    if (i < n) out[i] = sums[blockIdx.x] + sh[threadIdx.x] - v;
    if (i == n - 1) out[n] = sums[blockIdx.x] + sh[threadIdx.x];
}

// per segment: left count, children
__global__ void k_children(Level L)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= L.num_segs) return;
    const Seg sg = L.segs[s];
    const int count = sg.end - sg.begin;
    if (count == 1) { L.nl[s] = -1; return; }
    int nl = L.pre[sg.end] - L.pre[sg.begin];
    // everything on one side: the list keeps its order, first half / second half (KdTree.cpp:108-113)
    const bool degenerate = nl == 0 || nl == count;
    const int mid = degenerate ? sg.begin + count / 2 : sg.begin + nl;
    const int slot = atomicAdd(L.next_count, 2);
    Seg l, r;
    l.begin = sg.begin; l.end = mid; l.node = sg.node + 1;
    r.begin = mid; r.end = sg.end; r.node = sg.node + 2 * (mid - sg.begin);
    L.segs_next[slot] = l; L.segs_next[slot + 1] = r;
    atomicMax(L.max_count, max(mid - sg.begin, sg.end - mid));
    // encode for the scatter: nl < 0 => keep order; child slots
    L.nl[s] = degenerate ? -2 - slot : nl;
    L.axis[s] = slot;                      // (axis is no longer needed this level) child slot base
    L.mean[s] = __int_as_float(mid);
}

__global__ void k_scatter(Level L)
{
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= L.T) return;
    const int seg = L.seg_of_pos[pos];
    const int t = L.order[pos];
    if (seg < 0) { L.order_next[pos] = t; L.seg_of_pos_next[pos] = -1; return; }
    const int nl = L.nl[seg];
    if (nl == -1) { L.order_next[pos] = t; L.seg_of_pos_next[pos] = -1; return; }      // a leaf just emitted
    const Seg sg = L.segs[seg];
    const int slot = L.axis[seg];
    const int mid = __float_as_int(L.mean[seg]);
    int np = pos;
    if (nl >= 0)
    {
        const int left_before = L.pre[pos] - L.pre[sg.begin];
        np = L.flags[pos] ? sg.begin + left_before : sg.begin + nl + ((pos - sg.begin) - left_before);
    }
    L.order_next[np] = t;
    L.seg_of_pos_next[np] = np < mid ? slot : slot + 1;
}

struct Buf
{
    std::vector<void*> ptrs;
    ~Buf() { for (void* p : ptrs) cudaFree(p); }
    template <typename T> cudaError_t alloc(T** out, size_t n)
    {
        cudaError_t e = cudaMalloc((void**)out, (n ? n : 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(*out);
        return e;
    }
};

// The scratch block: level counters, then every per-triangle array of the build
struct Scratch
{
    int* counts;                                             // next_count, max_count, flag, -
    float *cx, *cy, *cz, *gx, *gy, *gz; int *order[2], *sop[2]; Seg* segs[2];
    unsigned long long *kmin, *kmax; float *mean, *big_sum; int *axis, *nl, *flags, *pre, *sums;
};

size_t carve(void* base, int T, Scratch* s)
{
    Scratch tmp;
    if (!s) s = &tmp;
    Carve c = { (char*)base, 0 };
    s->counts = c.take<int>(4);
    s->cx = c.take<float>(T); s->cy = c.take<float>(T); s->cz = c.take<float>(T);
    s->gx = c.take<float>(T); s->gy = c.take<float>(T); s->gz = c.take<float>(T);
    for (int k = 0; k < 2; k++) { s->order[k] = c.take<int>(T); s->sop[k] = c.take<int>(T); s->segs[k] = c.take<Seg>(T); }
    s->big_sum = c.take<float>(3 * (size_t)T);
    s->kmin = c.take<unsigned long long>(3 * (size_t)T); s->kmax = c.take<unsigned long long>(3 * (size_t)T);
    s->mean = c.take<float>(T); s->axis = c.take<int>(T); s->nl = c.take<int>(T);
    s->flags = c.take<int>(T); s->pre = c.take<int>((size_t)T + 1);
    s->sums = c.take<int>((size_t)(T + SCAN_BLOCK - 1) / SCAN_BLOCK + 1);
    return c.off;
}

} // namespace

#define BV_CUDA(call)                                                                       \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess)                                                              \
        {                                                                                   \
            rt_ctx_set_error(ctx, (std::string(#call) + ": " + cudaGetErrorString(e_)).c_str()); \
            return RT_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

size_t rt_bvh_scratch_bytes(int num_tris) { return carve(nullptr, num_tris, nullptr); }
int* rt_bvh_scratch_flag(void* scratch) { return (int*)scratch + 2; }

int rt_bvh_build_core(rt_gpu_ctx* ctx, const float* dP, const int* dI, int T, cudaStream_t st, void* scratch, int* host_counts,
                      rt_bvh_node* dnodes, rt_tri* dtris, int* out_depth)
{
    Scratch s;
    carve(scratch, T, &s);
    const int tb = 256, pg = (T + tb - 1) / tb;
    const int nb = (T + SCAN_BLOCK - 1) / SCAN_BLOCK;
    k_centroids<<<pg, tb, 0, st>>>(dP, dI, T, s.cx, s.cy, s.cz, s.order[0], s.sop[0]);
    const Seg root = { 0, T, 0 };
    BV_CUDA(cudaMemcpyAsync(s.segs[0], &root, sizeof root, cudaMemcpyHostToDevice, st));
    int num_segs = 1, depth = 0, cur = 0, level_max = T;
    while (num_segs > 0)
    {
        depth++;
        Level L;
        L.P = dP; L.I = dI; L.cx = s.cx; L.cy = s.cy; L.cz = s.cz; L.gx = s.gx; L.gy = s.gy; L.gz = s.gz;
        L.order = s.order[cur]; L.order_next = s.order[cur ^ 1];
        L.seg_of_pos = s.sop[cur]; L.seg_of_pos_next = s.sop[cur ^ 1];
        L.segs = s.segs[cur]; L.segs_next = s.segs[cur ^ 1];
        L.num_segs = num_segs; L.next_count = s.counts;
        L.kmin = s.kmin; L.kmax = s.kmax; L.mean = s.mean; L.axis = s.axis; L.nl = s.nl; L.flags = s.flags; L.pre = s.pre;
        L.nodes = dnodes; L.tris = dtris; L.T = T; L.big_sum = s.big_sum; L.max_count = s.counts + 1;
        BV_CUDA(cudaMemsetAsync(s.counts, 0, 2 * sizeof(int), st));
        k_init_keys<<<(3 * num_segs + tb - 1) / tb, tb, 0, st>>>(s.kmin, s.kmax, 3 * num_segs);
        k_bounds<<<pg, tb, 0, st>>>(L);
        k_gather<<<pg, tb, 0, st>>>(L);
        if (level_max > BIG_SEG) k_sum_big<<<num_segs, 64, 0, st>>>(L);
        k_nodes<<<(num_segs + 63) / 64, 64, 0, st>>>(L);
        k_flags<<<pg, tb, 0, st>>>(L);
        k_block_sums<<<nb, SCAN_BLOCK, 0, st>>>(s.flags, T, s.sums);
        k_scan_sums<<<1, SCAN_BLOCK, 0, st>>>(s.sums, nb);
        k_block_scan<<<nb, SCAN_BLOCK, 0, st>>>(s.flags, T, s.sums, s.pre);
        k_children<<<(num_segs + tb - 1) / tb, tb, 0, st>>>(L);
        k_scatter<<<pg, tb, 0, st>>>(L);
        BV_CUDA(cudaGetLastError());
        // one read per level: the next level's segment count and largest segment
        BV_CUDA(cudaMemcpyAsync(host_counts, s.counts, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
        BV_CUDA(cudaStreamSynchronize(st));
        num_segs = host_counts[0]; level_max = host_counts[1];
        cur ^= 1;
        if (depth > 4096) { rt_ctx_set_error(ctx, "rt_gpu_build_bvh: runaway depth"); return RT_ERR_CUDA; }
    }
    if (out_depth) *out_depth = depth;
    return RT_OK;
}

extern "C" int rt_gpu_build_bvh(rt_gpu_ctx* ctx, const float* points, int32_t num_points, const int32_t* indices,
                                int32_t num_tris, rt_bvh_node* out_nodes, rt_tri* out_tris, int32_t* out_depth, float* out_ms)
{
    if (!ctx) return RT_ERR_INVALID;
    if (!points || !indices || num_points <= 0 || num_tris <= 0 || !out_nodes || !out_tris)
    {
        rt_ctx_set_error(ctx, "rt_gpu_build_bvh: bad arguments");
        return RT_ERR_INVALID;
    }
    if ((long long)num_tris * 3 >= 0xFFFFFFFFll)
    {
        rt_ctx_set_error(ctx, "rt_gpu_build_bvh: too many triangles");
        return RT_ERR_INVALID;
    }
    for (long long k = 0; k < 3ll * num_tris; k++)
        if (indices[k] < 0 || indices[k] >= num_points)
        {
            rt_ctx_set_error(ctx, "rt_gpu_build_bvh: point index out of range");
            return RT_ERR_INVALID;
        }
    // a NaN or infinite coordinate is refused, as the upload and the mesh edits refuse it: the builder equals the host
    // builder on every input either of them accepts
    for (long long k = 0; k < 3ll * num_points; k++)
        if (!(fabsf(points[k]) <= FLT_MAX))
        {
            rt_ctx_set_error(ctx, "rt_gpu_build_bvh: non-finite point");
            return RT_ERR_INVALID;
        }
    BV_CUDA(cudaSetDevice(rt_ctx_device(ctx)));
    cudaStream_t st = (cudaStream_t)rt_gpu_stream(ctx);
    const int T = num_tris;
    Buf buf;
    float* dP; int* dI; char* scratch; rt_bvh_node* dnodes; rt_tri* dtris;
    BV_CUDA(buf.alloc(&dP, 3 * (size_t)num_points)); BV_CUDA(buf.alloc(&dI, 3 * (size_t)T));
    BV_CUDA(buf.alloc(&scratch, rt_bvh_scratch_bytes(T)));
    BV_CUDA(buf.alloc(&dnodes, 2 * (size_t)T)); BV_CUDA(buf.alloc(&dtris, T));
    BV_CUDA(cudaMemcpyAsync(dP, points, 3 * (size_t)num_points * sizeof(float), cudaMemcpyHostToDevice, st));
    BV_CUDA(cudaMemcpyAsync(dI, indices, 3 * (size_t)T * sizeof(int), cudaMemcpyHostToDevice, st));
    cudaEvent_t e0, e1;
    BV_CUDA(cudaEventCreate(&e0)); BV_CUDA(cudaEventCreate(&e1));
    BV_CUDA(cudaEventRecord(e0, st));
    int counts[4] = { 0, 0, 0, 0 }, depth = 0;
    const int rc = rt_bvh_build_core(ctx, dP, dI, T, st, scratch, counts, dnodes, dtris, &depth);
    if (rc != RT_OK) { cudaEventDestroy(e0); cudaEventDestroy(e1); return rc; }
    BV_CUDA(cudaEventRecord(e1, st));
    BV_CUDA(cudaMemcpyAsync(out_nodes, dnodes, (2 * (size_t)T - 1) * sizeof(rt_bvh_node), cudaMemcpyDeviceToHost, st));
    BV_CUDA(cudaMemcpyAsync(out_tris, dtris, (size_t)T * sizeof(rt_tri), cudaMemcpyDeviceToHost, st));
    BV_CUDA(cudaStreamSynchronize(st));
    float ms = 0.0f;
    BV_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (out_depth) *out_depth = depth;
    if (out_ms) *out_ms = ms;
    return RT_OK;
}
