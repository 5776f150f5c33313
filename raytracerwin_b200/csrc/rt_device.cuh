// rt_device.cuh — device-side arithmetic of the per-pixel ray/scene path (sm_100a).
//
// Everything here is compiled with -fmad=false and the default IEEE division / square root, so
// every fp32 operation rounds once, exactly like the reference's Linux build (no fast-math,
// CMakeLists.txt:27-29) compiled with -ffp-contract=off.  Each function names the reference code
// whose results it has to reproduce bit for bit (paths relative to the reference's Src/).
#pragma once

#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "rt_gpu.h"
#include "rt_rng.h"

namespace rtdev {

#define RT_FULL_MASK 0xffffffffu
#define RT_FLT_EPS 1.1920929e-07f           // FLT_EPSILON, MathHelper.h:12
#define RT_PI_REF 3.1415926f                // PI, MathHelper.h:14
#define RT_MAX_PATH_DEPTH 32                // deepest MaxBounceTimes the unwinding stack holds
#define RT_MAX_MATERIAL_DEPTH 8             // deepest nesting of Combine nodes

// ---- device copies of the scene -----------------------------------------------------------------
// All textures of a scene live in ONE float4 atlas (one cudaArray, one texture object: point
// sampling, unnormalised coordinates), so the texture handle is uniform across a warp whatever
// triangles its lanes hit; a DevTexture is the rectangle of one decoded PNG inside the atlas.
struct DevTexture
{
    int32_t x0, y0;             // origin inside the atlas
    int32_t width, height;
};

struct DevMesh
{
    const float4* nodes;        // 2 x float4 per rt_bvh_node: {bmin.xyz, escape} {bmax.xyz, tri}
    const float4* tris;         // 4 x float4 per rt_tri: {p0, index} {p1,-} {p2,-} {n,-}
    const float4* shade;        // 4 x float4 per rt_shade, in LEAF order on the device (record k <-> tris[k]; reordered at upload)
    const DevTexture* textures;
    const float4* octo;         // the tree collapsed to 8-wide nodes for the culled walk: 8 x {bmin.xyz, ref}{bmax.xyz, count}
                                // per node, children in slot order, ref = child node (>= 0) or ~leaf slot (see rt_walk_octo_kernel)
    int32_t num_nodes, num_tris, num_textures;
    float cull_scale;           // largest |coordinate| of the root bounds (culling margin)
};

struct DevScene
{
    const rt_shape* shapes;
    const rt_material* materials;
    const DevMesh* meshes;
    const rt_light* lights;
    cudaTextureObject_t atlas;  // every texture of the scene (see DevTexture); 0 when there is none
    const float4* unit_vectors; // PseudoRandomUnitVectors padded to 16 bytes
    uint32_t num_unit_vectors;
    int32_t num_shapes, num_materials, num_meshes, num_lights;
    float eye[3];
    float dir_z, ray_distance, bounce_offset;
    // Top of the first mesh's tree for the walk kernel's shared-memory stage: RT_TOP_SLOTS hashed slots,
    // top_tags[s] = node index held by slot s (or -1), top_nodes[2s..2s+1] = that node; built at upload from the
    // shallowest levels (breadth first).  top_of = the node array they belong to (other meshes bypass the stage).
    const int* top_tags;
    const float4* top_nodes;
    const float4* top_of;
};
#define RT_TOP_SLOTS 512
__host__ __device__ __forceinline__ unsigned top_slot(int node) { return ((unsigned)node * 0x9E3779B1u) >> 23; }

struct Ray { float3 o, d; float dist; };                                  // RRay, RRay.h:31-37
struct Hit { float3 pos, nrm; float dist; float3 color; float alpha; };   // RayHitResult, RRay.h:13-29
struct Rng { uint32_t key, n; };                                          // position in the rand() stream

struct Counters
{
    unsigned long long rays, camera_rays, shadow_rays, node_visits, tri_visits, mesh_hits, mesh_walks;
};

// ---- RVec3 arithmetic (RVector.h:97-234) --------------------------------------------------------
__device__ __forceinline__ float3 V3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 add3(float3 a, float3 b) { return V3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 sub3(float3 a, float3 b) { return V3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 mulf3(float3 a, float s) { return V3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float3 mul3(float3 a, float3 b) { return V3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float dot3(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }           // :207
__device__ __forceinline__ float3 cross3(float3 a, float3 b)                                                       // :213
{
    return V3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float magnitude3(float3 a) { return sqrtf(a.x * a.x + a.y * a.y + a.z * a.z); }        // :158
__device__ __forceinline__ bool eq_zero(float a) { return fabsf(a) < RT_FLT_EPS; }                                  // FLT_EQUAL_ZERO
__device__ __forceinline__ float min_ref(float a, float b) { return (a < b) ? a : b; }                              // Math::Min, MathHelper.h:38
__device__ __forceinline__ float max_ref(float a, float b) { return (a > b) ? a : b; }                              // Math::Max, MathHelper.h:35
__device__ __forceinline__ float3 ld3(const float* p) { return V3(p[0], p[1], p[2]); }
__device__ __forceinline__ float3 xyz(float4 v) { return V3(v.x, v.y, v.z); }

// One 32-byte record (a BVH node; half a leaf triangle) with ONE 256-bit load (LDG.E.256 on sm_100): a lane's node
// costs the L1 one request instead of two — the walk kernels are bound by exactly that (lanes at 32 different
// nodes).  Read-only path (.nc): the scene is immutable while rendering.  `p` is 32-byte aligned (cudaMalloc base,
// 32 / 64-byte records).
__device__ __forceinline__ void ld32(const float4* __restrict__ p, float4& a, float4& b)
{
#ifndef RT_NO_LDG256
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
#else
    a = __ldg(p); b = __ldg(p + 1);
#endif
}

// RVec3::GetNormalizedVec3, RVector.h:169-183 — short vectors are returned unchanged
__device__ __forceinline__ float3 normalized3(float3 a)
{
    float sqr_mag = a.x * a.x + a.y * a.y + a.z * a.z;
    if (!eq_zero(sqr_mag))
    {
        float one_over_mag = 1.0f / sqrtf(sqr_mag);
        return V3(a.x * one_over_mag, a.y * one_over_mag, a.z * one_over_mag);
    }
    return a;
}

// Math::Q_rsqrt, MathHelper.cpp:26-38 (magic constant, one Newton step)
__device__ __forceinline__ float q_rsqrt(float number)
{
    const float x2 = number * 0.5F;
    uint32_t i = __float_as_uint(number);
    i = 0x5f3759df - (i >> 1);
    float y = __uint_as_float(i);
    y = y * (1.5F - (x2 * y * y));
    return y;
}

// RVec3::GetNormalizedVec3_Fast, RVector.h:185-199
__device__ __forceinline__ float3 normalized_fast3(float3 a)
{
    float sqr_mag = a.x * a.x + a.y * a.y + a.z * a.z;
    if (!eq_zero(sqr_mag))
    {
        float one_over_mag = q_rsqrt(sqr_mag);
        return V3(a.x * one_over_mag, a.y * one_over_mag, a.z * one_over_mag);
    }
    return a;
}

// RVec3::Reflect, RVector.h:218-221: *this - normal * 2.0f * Dot(*this, normal)
__device__ __forceinline__ float3 reflect3(float3 v, float3 n) { return sub3(v, mulf3(mulf3(n, 2.0f), dot3(v, n))); }

__device__ __forceinline__ float rng_random(Rng& r) { return rt_random01(r.key, r.n++); }     // RMath::Random, Math.h:17-20
__device__ __forceinline__ int32_t rng_rand(Rng& r) { return rt_rand31(r.key, r.n++); }

__device__ __forceinline__ bool finite3(float3 a)
{
    return (fabsf(a.x) <= FLT_MAX) && (fabsf(a.y) <= FLT_MAX) && (fabsf(a.z) <= FLT_MAX);
}

// ---- ray/box ------------------------------------------------------------------------------------
// Per-ray constants of RRay::TestIntersectionWithAabb (RRay.cpp:89-136): the reference recomputes
// 1.0f / Direction per box; the quotient is the same every time, so it is formed once per ray.
struct RayPre
{
    float3 inv;         // 1/d on enabled axes
    bool ex, ey, ez;    // axis enabled: !FLT_EQUAL_ZERO(d)
    float cull_pad;     // t-space margin of the culled traversal (see bvh_traverse)
};

__device__ __forceinline__ RayPre ray_pre(const Ray& r)
{
    RayPre p;
    p.ex = !eq_zero(r.d.x); p.ey = !eq_zero(r.d.y); p.ez = !eq_zero(r.d.z);
    p.inv.x = p.ex ? 1.0f / r.d.x : 0.0f;
    p.inv.y = p.ey ? 1.0f / r.d.y : 0.0f;
    p.inv.z = p.ez ? 1.0f / r.d.z : 0.0f;
    p.cull_pad = 0.0f;
    return p;
}

// The reference test verbatim (any direction, NaN and infinities included): a LINE test,
// accept iff tmax > tmin; tlo/thi return the clipped interval.
__device__ __forceinline__ bool slab_general(const Ray& r, const RayPre& p, float3 bmin, float3 bmax, float& tlo, float& thi)
{
    float tmin = -FLT_MAX, tmax = FLT_MAX;
    if (p.ex)
    {
        float t1 = (bmin.x - r.o.x) * p.inv.x, t2 = (bmax.x - r.o.x) * p.inv.x;
        tmin = max_ref(tmin, min_ref(t1, t2)); tmax = min_ref(tmax, max_ref(t1, t2));
    }
    if (p.ey)
    {
        float t1 = (bmin.y - r.o.y) * p.inv.y, t2 = (bmax.y - r.o.y) * p.inv.y;
        tmin = max_ref(tmin, min_ref(t1, t2)); tmax = min_ref(tmax, max_ref(t1, t2));
    }
    if (p.ez)
    {
        float t1 = (bmin.z - r.o.z) * p.inv.z, t2 = (bmax.z - r.o.z) * p.inv.z;
        tmin = max_ref(tmin, min_ref(t1, t2)); tmax = min_ref(tmax, max_ref(t1, t2));
    }
    tlo = tmin; thi = tmax;
    return tmax > tmin;
}

// Same result when all three axes are enabled and origin/direction are finite (then no NaN can
// arise for finite boxes and fminf/fmaxf equal the reference's ternaries): branch-free FMNMX form.
__device__ __forceinline__ bool slab_fast(const Ray& r, const RayPre& p, float3 bmin, float3 bmax, float& tlo, float& thi)
{
    float x1 = (bmin.x - r.o.x) * p.inv.x, x2 = (bmax.x - r.o.x) * p.inv.x;
    float y1 = (bmin.y - r.o.y) * p.inv.y, y2 = (bmax.y - r.o.y) * p.inv.y;
    float z1 = (bmin.z - r.o.z) * p.inv.z, z2 = (bmax.z - r.o.z) * p.inv.z;
    float tmin = fmaxf(fmaxf(fmaxf(-FLT_MAX, fminf(x1, x2)), fminf(y1, y2)), fminf(z1, z2));
    float tmax = fminf(fminf(fminf(FLT_MAX, fmaxf(x1, x2)), fmaxf(y1, y2)), fmaxf(z1, z2));
    tlo = tmin; thi = tmax;
    return tmax > tmin;
}

// ---- ray/triangle -------------------------------------------------------------------------------
// RRay::TestIntersectionWithTriangleAndFaceNormal, RRay.cpp:147-213, with the face normal the
// host precomputed exactly as RRay.cpp:138-145 derives it per test.
__device__ __forceinline__ bool triangle_test(const Ray& r, float3 p0, float3 p1, float3 p2, float3 n,
                                              float3& pos, float& dist)
{
    float3 end = add3(r.o, mulf3(r.d, r.dist));
    float d0 = dot3(n, r.o);
    float d1 = dot3(n, p0);
    float d2 = d0 - d1;
    if (d2 < 0) return false;
    if (dot3(end, n) - d1 > 0) return false;
    float3 l = sub3(end, r.o);
    float d3 = dot3(n, l);
    if (eq_zero(d3)) return false;
    float df = -(d2 / d3);
    float3 cp = add3(r.o, mulf3(l, df));
    if (dot3(cross3(sub3(p1, p0), n), sub3(cp, p0)) > 0) return false;
    if (dot3(cross3(sub3(p2, p1), n), sub3(cp, p1)) > 0) return false;
    if (dot3(cross3(sub3(p0, p2), n), sub3(cp, p2)) > 0) return false;
    pos = cp;
    dist = magnitude3(mulf3(l, df));
    return true;
}

// RRay::TestIntersectionWithSphere, RRay.cpp:25-64
__device__ __forceinline__ bool sphere_test(const Ray& r, float3 c, float radius, float3& pos, float3& nrm, float& dist)
{
    float dx = r.d.x * r.dist, dy = r.d.y * r.dist, dz = r.d.z * r.dist;
    float _a = dx * dx + dy * dy + dz * dz;
    float _b = 2 * dx * (r.o.x - c.x) + 2 * dy * (r.o.y - c.y) + 2 * dz * (r.o.z - c.z);
    float _c = c.x * c.x + c.y * c.y + c.z * c.z + r.o.x * r.o.x + r.o.y * r.o.y + r.o.z * r.o.z +
               -2 * (c.x * r.o.x + c.y * r.o.y + c.z * r.o.z) - radius * radius;
    float d = _b * _b - 4 * _a * _c;
    if (d >= 0)
    {
        float t = (-_b - sqrtf(d)) / (_a * 2);
        if (t <= 0) return false;
        float3 hp = V3(r.o.x + t * dx, r.o.y + t * dy, r.o.z + t * dz);
        float dd = magnitude3(sub3(hp, r.o));
        if (dd > r.dist) return false;
        pos = hp; nrm = normalized3(sub3(hp, c)); dist = dd;
        return true;
    }
    return false;
}

// RRay::TestIntersectionWithPlane, RRay.cpp:66-87 (the 1e-6 literal is a double in the reference)
__device__ __forceinline__ bool plane_test(const Ray& r, float3 n, float3 p, float3& pos, float3& nrm, float& dist)
{
    float denom = dot3(n, r.d);
    if ((double)fabsf(denom) > 1e-6)
    {
        float3 p0l0 = sub3(p, r.o);
        float t = dot3(p0l0, n) / denom;
        if (t >= 0 && t < r.dist)
        {
            pos = add3(r.o, mulf3(r.d, t)); nrm = n; dist = t;
            return true;
        }
    }
    return false;
}

// RCapsule::TestRayCylinderIntersection, Shapes.cpp:65-125 (no comparison with the ray length)
__device__ __forceinline__ bool cylinder_test(const Ray& r, float3 start, float3 endp, float radius,
                                              float3& pos, float3& nrm, float& dist)
{
    float3 d = sub3(endp, start);
    float3 m = sub3(r.o, start);
    float dd = dot3(d, d), nd = dot3(r.d, d), mn = dot3(m, r.d), md = dot3(m, d), mm = dot3(m, m);
    if (dot3(sub3(r.o, start), sub3(endp, start)) < 0 && dot3(r.d, sub3(endp, start)) < 0) return false;
    if (dot3(sub3(r.o, endp), sub3(start, endp)) < 0 && dot3(r.d, sub3(start, endp)) < 0) return false;
    float a = dd - nd * nd;
    float b = dd * mn - nd * md;
    float c = dd * (mm - radius * radius) - md * md;
    if (fabsf(a) < RT_FLT_EPS) return false;
    if ((b * b - a * c) < 0) return false;
    float r_t = (-b - sqrtf(b * b - a * c)) / a;
    if (r_t < 0) return false;
    float3 v = add3(r.o, mulf3(r.d, r_t));
    if (dot3(sub3(v, start), sub3(endp, start)) < 0) return false;
    if (dot3(sub3(v, endp), sub3(start, endp)) < 0) return false;
    dist = r_t;
    pos = add3(r.o, mulf3(r.d, r_t));
    float3 side = cross3(sub3(endp, start), sub3(pos, start));
    nrm = normalized3(cross3(side, sub3(endp, start)));
    return true;
}

// RMath::Barycentric, Math.cpp:56-68
__device__ __forceinline__ void barycentric(float3 p, float3 a, float3 b, float3 c, float& u, float& v, float& w)
{
    float3 v0 = sub3(b, a), v1 = sub3(c, a), v2 = sub3(p, a);
    float d00 = dot3(v0, v0), d01 = dot3(v0, v1), d11 = dot3(v1, v1), d20 = dot3(v2, v0), d21 = dot3(v2, v1);
    float denom = d00 * d11 - d01 * d01;
    v = (d11 * d20 - d01 * d21) / denom;
    w = (d00 * d21 - d01 * d20) / denom;
    u = 1.0f - v - w;
}

__device__ __forceinline__ float lerp_ref(float a, float b, float t) { return a + (b - a) * t; }   // Math::Lerp, MathHelper.h:40

// (int)f as the reference's x86 build evaluates it (cvttss2si: INT_MIN for NaN / out of range)
__device__ __forceinline__ int to_int_ref(float f)
{
    if (!(f > -2147483904.0f && f < 2147483648.0f)) return INT32_MIN;
    return (int)f;
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// RTexture::Sample, Texture.cpp:23-57: repeat addressing, (W-1,H-1) scaling, floor/ceil taps and
// three fp32 lerps done by hand — the texture unit only fetches texels (point mode), because its
// own bilinear filter uses 8-bit weights and a half-texel convention.  Texel indices are clamped
// into the image where the reference would read out of bounds (NaN uv).
__device__ __forceinline__ float4 texture_sample(cudaTextureObject_t atlas, const DevTexture& t, float u, float v)
{
    float cu = u - floorf(u), cv = v - floorf(v);
    float fx = cu * (float)(t.width - 1), fy = cv * (float)(t.height - 1);
    int x0 = to_int_ref(floorf(fx)), y0 = to_int_ref(floorf(fy));
    int x1 = to_int_ref(ceilf(fx)), y1 = to_int_ref(ceilf(fy));
    float dx = fx - (float)x0, dy = fy - (float)y0;
    float cx0 = (float)(t.x0 + clampi(x0, 0, t.width - 1)) + 0.5f, cx1 = (float)(t.x0 + clampi(x1, 0, t.width - 1)) + 0.5f;
    float cy0 = (float)(t.y0 + clampi(y0, 0, t.height - 1)) + 0.5f, cy1 = (float)(t.y0 + clampi(y1, 0, t.height - 1)) + 0.5f;
    float4 p00 = tex2D<float4>(atlas, cx0, cy0);
    float4 p01 = tex2D<float4>(atlas, cx1, cy0);
    float4 p10 = tex2D<float4>(atlas, cx0, cy1);
    float4 p11 = tex2D<float4>(atlas, cx1, cy1);
    float4 o;
    o.x = lerp_ref(lerp_ref(p00.x, p01.x, dx), lerp_ref(p10.x, p11.x, dx), dy);
    o.y = lerp_ref(lerp_ref(p00.y, p01.y, dx), lerp_ref(p10.y, p11.y, dx), dy);
    o.z = lerp_ref(lerp_ref(p00.z, p01.z, dx), lerp_ref(p10.z, p11.z, dx), dy);
    o.w = lerp_ref(lerp_ref(p00.w, p01.w, dx), lerp_ref(p10.w, p11.w, dx), dy);
    return o;
}

// ---- mesh hit attributes ---------------------------------------------------------------------------
// RMeshShape::TestRayIntersection after the tree walk (MeshShape.cpp:286-326): barycentrics,
// Q_rsqrt-normalised interpolated normal, uv interpolation, texture sample.  The whole record is
// replaced (KdTree.cpp:178-181 assigns a fresh RayHitResult: colour 1, alpha 1).
__device__ __forceinline__ void mesh_attributes(cudaTextureObject_t atlas, const DevMesh& m, int slot, float3 pos, float dist, Hit& out, int& tri_index)
{
    float4 t0, t1, s0, s1, s2, s3;
    ld32(m.tris + 4 * (size_t)slot, t0, t1);
    const float4 t2 = __ldg(m.tris + 4 * (size_t)slot + 2);
    // rt_shade: n0[3] n1[3] n2[3] uv0[2] uv1[2] uv2[2] texture
    ld32(m.shade + 4 * (size_t)slot, s0, s1);               // n0.xyz n1.x | n1.yz n2.xy
    ld32(m.shade + 4 * (size_t)slot + 2, s2, s3);           // n2.z uv0.xy uv1.x | uv1.y uv2.xy texture
    const int index = __float_as_int(t0.w);
    tri_index = index;
    out.pos = pos; out.dist = dist;
    out.color = V3(1.0f, 1.0f, 1.0f); out.alpha = 1.0f;
    float u, v, w;
    barycentric(pos, xyz(t0), xyz(t1), xyz(t2), u, v, w);
    const float3 n0 = V3(s0.x, s0.y, s0.z), n1 = V3(s0.w, s1.x, s1.y), n2 = V3(s1.z, s1.w, s2.x);
    float3 nn = add3(add3(mulf3(n0, u), mulf3(n1, v)), mulf3(n2, w));
    out.nrm = normalized_fast3(nn);
    const int texture = __float_as_int(s3.w);
    if (texture >= 0)
    {
        // t0*u + t1*v + t2*w, then Sample(x, 1 - y)  (MeshShape.cpp:316-324)
        float tx = s2.y * u + s2.w * v + s3.y * w;
        float ty = s2.z * u + s3.x * v + s3.z * w;
        const DevTexture tex = m.textures[texture];
        float4 c = texture_sample(atlas, tex, tx, 1.0f - ty);
        out.color = V3(c.x, c.y, c.z);
        out.alpha = c.w;
    }
}

// ---- mesh: BVH traversal + hit attributes ---------------------------------------------------------
// KdNode::TestRayIntersection (KdTree.cpp:128-195) on the pre-order, escape-threaded node array:
// a node whose slab test passes continues at i+1 (Left, then Right in pre-order); a rejected
// node or a finished leaf jumps to `escape`.  Ray.dist shrinks at every accepted leaf (:176) and
// the LAST accepted leaf in this fixed order wins (:178-186), exactly as in the reference.
//
// CULL (RT_TRAVERSE_CULLED) additionally skips a subtree when no triangle inside its box can be
// accepted.  An accepted hit has cp = O + (End-O)*df inside the triangle's prism and within
// rounding of its plane, i.e. inside the leaf box grown by a few ulps of the coordinates, with
// df in [0, 1+] — so the line parameter t = dist*df lies inside the box's slab interval widened
// by that growth divided by |d| on each axis.  With pad = growth * max|1/d| over the enabled axes
// the subtree is skipped iff  thi < -pad  or  tlo > dist*(1+2^-7) + pad.  Order, the evolving
// dist and every accepted hit are the same as in the exact walk; only rejected work is dropped.
// ANY (shadow queries, RayTracerScene.cpp:152-164) stops at the first accepted triangle when
// CULL is on: the reference keeps walking but only the boolean is used.
//
// Rays that run nearly parallel to an axis (|1/d| large on it) would make that single pad so wide
// that nothing is culled; for them (`wide`) the interval is padded per axis instead (cull_axes):
// each slab's own interval is widened by growth * |1/d_axis| before the three are intersected,
// which is the same bound, just not collapsed to its worst axis.
//
// The walk is RESUMABLE: its whole state is a node cursor plus the best hit so far, kept per lane
// in a Query.  A warp runs rounds of "node steps until every walking lane holds a leaf, then the
// triangle tests of those leaves together", and leaves the loop as soon as fewer than `min_lanes`
// lanes are still walking, so the caller can hand the idle lanes new rays and come back — the
// slow lanes keep their cursor.  That is what keeps the 32 lanes of a warp busy although one ray
// may visit 3 nodes and its neighbour 3000.
enum { ST_IDLE = 0, ST_SHAPES = 1, ST_TRAVERSE = 2, ST_MESHDONE = 3, ST_SHADE = 4 };

// per-axis form of the culling interval; true = no triangle in this box can be accepted
// On a DISABLED axis (|d| < FLT_EPSILON: the reference skips that slab, RRay.cpp:95,105,115) the ray moves
// less than FLT_EPSILON * Distance, so an accepted hit — a point inside its triangle, hence inside the box —
// needs the box to contain the origin's coordinate within `slack` = growth + FLT_EPSILON * Distance.
__device__ __forceinline__ bool cull_axes(const Ray& r, const RayPre& p, float3 pad3, float3 bmin, float3 bmax, float dist_hi, float growth)
{
    const float slack = growth + RT_FLT_EPS * dist_hi;
    if (!p.ex && (r.o.x < bmin.x - slack || r.o.x > bmax.x + slack)) return true;
    if (!p.ey && (r.o.y < bmin.y - slack || r.o.y > bmax.y + slack)) return true;
    if (!p.ez && (r.o.z < bmin.z - slack || r.o.z > bmax.z + slack)) return true;
    const float x1 = (bmin.x - r.o.x) * p.inv.x, x2 = (bmax.x - r.o.x) * p.inv.x;
    const float y1 = (bmin.y - r.o.y) * p.inv.y, y2 = (bmax.y - r.o.y) * p.inv.y;
    const float z1 = (bmin.z - r.o.z) * p.inv.z, z2 = (bmax.z - r.o.z) * p.inv.z;
    const float lo = fmaxf(fmaxf(fminf(x1, x2) - pad3.x, fminf(y1, y2) - pad3.y), fminf(z1, z2) - pad3.z);
    const float hi = fminf(fminf(fmaxf(x1, x2) + pad3.x, fmaxf(y1, y2) + pad3.y), fmaxf(z1, z2) + pad3.z);
    return hi < 0.0f || lo > dist_hi;
}

// growth of the leaf boxes that covers the rounding of cp: 2^-16 of the coordinate scale
__device__ __forceinline__ float cull_growth(const Ray& r, float mesh_scale)
{
    return (fmaxf(fmaxf(fabsf(r.o.x), fabsf(r.o.y)), fabsf(r.o.z)) + mesh_scale) * 1.52587890625e-05f;
}

// t-space margin of the culled walk: growth of the leaf boxes that covers the rounding of cp
// (2^-16 of the coordinate scale), converted to the ray parameter by the largest |1/d|
__device__ __forceinline__ float cull_pad_for(const Ray& r, const RayPre& pre, float mesh_scale)
{
    const float scale = fmaxf(fmaxf(fabsf(r.o.x), fabsf(r.o.y)), fabsf(r.o.z)) + mesh_scale;
    const float growth = scale * 1.52587890625e-05f;
    const float mi_x = pre.ex ? fabsf(pre.inv.x) : 0.0f, mi_y = pre.ey ? fabsf(pre.inv.y) : 0.0f, mi_z = pre.ez ? fabsf(pre.inv.z) : 0.0f;
    float pad = growth * fmaxf(fmaxf(mi_x, mi_y), mi_z) + growth;
    // NaN/inf: never cull.  Nor with a negative Distance (a bounce after a hit beyond the segment's end: the
    // capsule test does not compare with Distance, and |d| > 1 makes a triangle's distance exceed it): the reference
    // then accepts triangles BEHIND the origin, and an accepted hit makes Distance positive again
    if (!(pad <= FLT_MAX) || !(r.dist >= 0.0f)) pad = FLT_MAX;
    return pad;
}

struct Query
{
    Ray r;              // TestRay of FindIntersectionWithScene: r.dist shrinks as hits are accepted
    RayPre pre;
    Hit h;              // the RayHitResult the shapes write into (stale fields survive, Appendix A11)
    float3 bpos;        // position of the last accepted triangle of the mesh being walked
    int si;             // shape cursor (insertion order = test order)
    int node;           // node cursor inside the current mesh
    int best;           // leaf slot of the last accepted triangle, -1 = none yet
    int hit_shape, tri; // result: shape index (nearest) / 0 (any) / -1, original triangle id
    bool any;           // shadow query: any accepted hit
    bool weird;         // a disabled slab axis or a non-finite component: use the verbatim slab test
};

__device__ __forceinline__ void query_begin(Query& q, const Ray& ray, bool any, Counters& cnt)
{
    q.r = ray;
    q.pre = ray_pre(ray);
    q.weird = !(q.pre.ex && q.pre.ey && q.pre.ez && finite3(ray.o) && finite3(ray.d));
    q.h.pos = V3(0, 0, 0); q.h.nrm = V3(0, 0, 0); q.h.dist = 0.0f; q.h.color = V3(1.0f, 1.0f, 1.0f); q.h.alpha = 1.0f;
    q.bpos = V3(0, 0, 0);
    q.si = 0; q.node = 0; q.best = -1; q.hit_shape = -1; q.tri = -1;
    q.any = any;
    cnt.rays++;
    if (any) cnt.shadow_rays++;
}

// Warp-collective.  Lanes with state == ST_TRAVERSE walk sc.meshes[shapes[q.si].mesh]; a lane that
// finishes its tree becomes ST_MESHDONE.  Returns when fewer than min_lanes (>= 1) lanes walk.
template <bool CULL>
__device__ __forceinline__ void query_traverse(const DevScene& sc, Query& q, int& state, int min_lanes, int leaf_wait, Counters& cnt)
{
    if (__ballot_sync(RT_FULL_MASK, state == ST_TRAVERSE) == 0) return;
    const float4* __restrict__ nodes = nullptr;
    const float4* __restrict__ tris = nullptr;
    int n = 0;
    if (state == ST_TRAVERSE)
    {
        const DevMesh* m = sc.meshes + sc.shapes[q.si].mesh;
        nodes = m->nodes; tris = m->tris; n = m->num_nodes;
    }
    const bool verbatim = __any_sync(RT_FULL_MASK, state == ST_TRAVERSE && q.weird);
    unsigned nodes_seen = 0, tris_seen = 0;
    int i = q.node;
    for (;;)
    {
        int leaf = -1;
        // node steps until every walking lane holds a leaf (or ran off its tree)
        for (;;)
        {
            const bool step = state == ST_TRAVERSE && leaf < 0 && i < n;
            const unsigned stepping = __ballot_sync(RT_FULL_MASK, step);
            if (stepping == 0) break;
            // do not let a few long walks hold many found leaves: test the leaves once the walkers
            // are fewer than the lanes that wait with one
            if (leaf_wait > 0 && __popc(__ballot_sync(RT_FULL_MASK, leaf >= 0)) >= leaf_wait && __popc(stepping) < leaf_wait) break;
            if (step)
            {
                float4 a, b;
                ld32(nodes + 2 * (size_t)i, a, b);
                const int escape = __float_as_int(a.w);
                const int tri = __float_as_int(b.w);
                nodes_seen++;
                float tlo, thi;
                bool enter = verbatim ? slab_general(q.r, q.pre, xyz(a), xyz(b), tlo, thi)
                                      : slab_fast(q.r, q.pre, xyz(a), xyz(b), tlo, thi);
                if (CULL) enter = enter && !(thi < -q.pre.cull_pad) && !(tlo > q.r.dist * 1.0078125f + q.pre.cull_pad);
                if (!enter) i = escape;
                else if (tri < 0) i = i + 1;
                else { leaf = tri; i = escape; }
            }
        }
        // the triangle tests of this round, together
        if (leaf >= 0)
        {
            float4 t0, t1, t2, t3;
            ld32(tris + 4 * (size_t)leaf, t0, t1);
            ld32(tris + 4 * (size_t)leaf + 2, t2, t3);
            tris_seen++;
            float3 hp; float hd;
            if (triangle_test(q.r, xyz(t0), xyz(t1), xyz(t2), xyz(t3), hp, hd))
            {
                q.r.dist = hd;
                q.bpos = hp;
                q.best = leaf;
                if (CULL && q.any) i = n;
            }
        }
        if (state == ST_TRAVERSE && i >= n) state = ST_MESHDONE;
        if (__popc(__ballot_sync(RT_FULL_MASK, state == ST_TRAVERSE)) < min_lanes) break;
    }
    q.node = i;
    cnt.node_visits += nodes_seen;
    cnt.tri_visits += tris_seen;
}

// ---- scene: nearest hit / any hit -------------------------------------------------------------------
// RayTracerScene::FindIntersectionWithScene (RayTracerScene.cpp:99-125) when q.any == false, the
// shadow loop of CalculateLightColor (:152-164) when q.any == true, cut into resumable pieces:
//   query_shapes    walks the shape list from q.si: bounds test, analytic shapes inline; stops at
//                   a mesh whose bounds the ray enters (state -> ST_TRAVERSE) or at the end of the
//                   list / the first shadow hit (state -> ST_SHADE);
//   query_traverse  (above) walks that mesh;
//   query_mesh_done turns the walk's result into the RayHitResult (attributes) and moves on.
// `q.h` is written the way the reference's shapes write RayHitResult: spheres, planes and the
// capsule's cylinder leave colour/alpha alone.
template <bool CULL>
__device__ __forceinline__ void query_shapes(const DevScene& sc, Query& q, int& state, Counters& cnt)
{
    while (state == ST_SHAPES)
    {
        if (q.si >= sc.num_shapes) { state = ST_SHADE; break; }
        const rt_shape* sh = sc.shapes + q.si;
        const int type = sh->type;
        bool enter = true;
        if (sh->has_bounds)
        {
            float tlo, thi;
            cnt.node_visits++;
            enter = slab_general(q.r, q.pre, ld3(sh->bounds_min), ld3(sh->bounds_max), tlo, thi);
        }
        if (type == RT_SHAPE_MESH)
        {
            const int mi = sh->mesh;
            if (enter && mi >= 0 && sc.meshes[mi].num_nodes > 0)
            {
                if (CULL) q.pre.cull_pad = cull_pad_for(q.r, q.pre, sc.meshes[mi].cull_scale);
                q.node = 0; q.best = -1;
                state = ST_TRAVERSE;
                cnt.mesh_walks++;           // one KdTree::TestRayIntersection call (MeshShape.cpp:284)
                break;
            }
            q.si++;
            continue;
        }
        bool hit = false;
        if (enter)
        {
            float3 pos = V3(0, 0, 0), nrm = V3(0, 0, 0); float dist = 0.0f;
            if (type == RT_SHAPE_SPHERE)                                  // Shapes.cpp:18-21
            {
                hit = sphere_test(q.r, ld3(sh->a), sh->radius, pos, nrm, dist);
                if (hit) { q.h.pos = pos; q.h.nrm = nrm; q.h.dist = dist; }
            }
            else if (type == RT_SHAPE_PLANE)                              // Shapes.cpp:23-26
            {
                hit = plane_test(q.r, ld3(sh->a), ld3(sh->b), pos, nrm, dist);
                if (hit) { q.h.pos = pos; q.h.nrm = nrm; q.h.dist = dist; }
            }
            else if (type == RT_SHAPE_TRIANGLE)                           // Shapes.cpp:127-130
            {
                const float3 p0 = ld3(sh->a), p1 = ld3(sh->b), p2 = ld3(sh->c);
                const float3 n = normalized3(cross3(sub3(p1, p0), sub3(p2, p0)));   // RRay.cpp:138-145
                hit = triangle_test(q.r, p0, p1, p2, n, pos, dist);
                if (hit) { q.h.pos = pos; q.h.nrm = n; q.h.dist = dist; }
            }
            else if (type == RT_SHAPE_CAPSULE)                            // Shapes.cpp:34-63
            {
                if (cylinder_test(q.r, ld3(sh->a), ld3(sh->b), sh->radius, pos, nrm, dist))
                {
                    hit = true;
                    q.h.dist = dist; q.h.pos = pos; q.h.nrm = nrm;
                }
                else
                {
                    float3 p1, n1, p2, n2; float d1 = 0.0f, d2 = 0.0f;
                    const bool b1 = sphere_test(q.r, ld3(sh->a), sh->radius, p1, n1, d1);
                    const bool b2 = sphere_test(q.r, ld3(sh->b), sh->radius, p2, n2, d2);
                    hit = b1 || b2;
                    if (hit)
                    {
                        const bool first = (b1 && b2) ? (d1 < d2) : b1;
                        // whole-struct assignment from a fresh RayHitResult: colour/alpha reset to 1
                        q.h.pos = first ? p1 : p2; q.h.nrm = first ? n1 : n2; q.h.dist = first ? d1 : d2;
                        q.h.color = V3(1.0f, 1.0f, 1.0f); q.h.alpha = 1.0f;
                    }
                }
            }
        }
        if (hit)
        {
            if (q.any) { q.hit_shape = 0; state = ST_SHADE; break; }     // `break` of the shadow loop
            q.r.dist = q.h.dist; q.hit_shape = q.si; q.tri = -1;
        }
        q.si++;
    }
}

// lanes whose walk ended (ST_MESHDONE): RMeshShape::TestRayIntersection's tail (MeshShape.cpp:286-326)
__device__ __forceinline__ void query_mesh_done(const DevScene& sc, Query& q, int& state, Counters& cnt)
{
    if (state != ST_MESHDONE) return;
    state = ST_SHAPES;
    if (q.best >= 0)
    {
        if (q.any) { q.hit_shape = 0; state = ST_SHADE; return; }
        const DevMesh m = sc.meshes[sc.shapes[q.si].mesh];
        mesh_attributes(sc.atlas, m, q.best, q.bpos, q.r.dist, q.h, q.tri);
        cnt.mesh_hits++;
        q.hit_shape = q.si;            // r.dist already equals h.dist (KdTree.cpp:176, RayTracerScene.cpp:117)
    }
    q.si++;
}

// One whole query, run to completion by the calling warp (test hooks; all lanes must call).
template <bool CULL>
__device__ __forceinline__ int trace_scene(const DevScene& sc, const Ray& in, bool active, bool any,
                                           Hit& h, int& tri_out, Counters& cnt)
{
    Query q;
    int state = ST_IDLE;
    if (active) { query_begin(q, in, any, cnt); state = ST_SHAPES; }
    else { q.r = in; q.pre = ray_pre(in); q.weird = false; q.h = h; q.bpos = V3(0, 0, 0); q.si = 0; q.node = 0; q.best = -1; q.hit_shape = -1; q.tri = -1; q.any = any; }
    for (;;)
    {
        query_shapes<CULL>(sc, q, state, cnt);
        if (__ballot_sync(RT_FULL_MASK, state == ST_TRAVERSE) == 0) break;
        query_traverse<CULL>(sc, q, state, 1, 0, cnt);
        query_mesh_done(sc, q, state, cnt);
    }
    if (active) { h = q.h; tri_out = q.tri; }
    return q.hit_shape;
}

// ---- materials ----------------------------------------------------------------------------------------
struct Bounce { float3 att, emi; };                                        // ViewRayBounceResult

// RMath::RandomUnitVector, Math.h:34-40.  sinf/cosf/acosf are CUDA's, not glibc's: results may
// differ from the CPU in the last ulp (the only non-bit-exact arithmetic on the path).
__device__ __forceinline__ float3 random_unit_vector(Rng& rng)
{
    float t1 = 2.0f * RT_PI_REF * rng_random(rng);
    float t2 = acosf(1.0f - 2.0f * rng_random(rng));
    float sin_t2 = sinf(t2);
    return V3(sinf(t1) * sin_t2, cosf(t1) * sin_t2, cosf(t2));
}

// RMath::RandomHemisphereDirection, Math.cpp:42-54, table index drawn from the counter RNG
// (the reference's shared cursor, Math.cpp:33-40, is replaced on both sides; see include/rt_rng.h)
__device__ __forceinline__ float3 random_hemisphere(const DevScene& sc, float3 n, Rng& rng)
{
    uint32_t idx = (uint32_t)rng_rand(rng) % sc.num_unit_vectors;
    float3 v = xyz(__ldg(sc.unit_vectors + idx));
    if (dot3(v, n) > 0.0f) return v;
    return reflect3(v, n);
}

// SurfaceMaterial_DiffuseChecker::IsBrighterArea, SurfaceMaterials.cpp:66-90
__device__ __forceinline__ bool checker_bright(float3 p, float recip)
{
    bool r = false;
    float fx = p.x * recip, fy = p.y * recip, fz = p.z * recip;
    if (fx - floorf(fx) > 0.5f) r = !r;
    if (fz - floorf(fz) > 0.5f) r = !r;
    if (fy - floorf(fy) > 0.5f) r = !r;
    return r;
}

// One leaf material: BounceViewRay (preview == false) or PreviewColor (preview == true, colour
// returned in .att).  SurfaceMaterials.cpp:20-38,53-64,98-125,132-143,179-192.
__device__ __forceinline__ Bounce material_leaf(const DevScene& sc, const rt_material& m, bool preview,
                                                const Ray& in, const Hit& h, Ray& out, Rng& rng)
{
    Bounce r; r.att = V3(0, 0, 0); r.emi = V3(0, 0, 0);
    const float3 rgb = V3(m.rgb[0], m.rgb[1], m.rgb[2]);
    if (m.type == RT_MAT_DIFFUSE || m.type == RT_MAT_CHECKER)
    {
        float factor = 1.0f;
        if (m.type == RT_MAT_CHECKER) factor = checker_bright(h.pos, m.scalar) ? 1.0f : 0.5f;
        if (preview)
        {
            r.att = mulf3(rgb, dot3(h.nrm, V3(0, 1, 0)) * 0.5f + 0.5f);
            if (m.type == RT_MAT_CHECKER) r.att = mulf3(r.att, factor);
            return r;
        }
        float remaining = in.dist - h.dist;
        float3 dir = random_hemisphere(sc, h.nrm, rng);
        out.o = add3(h.pos, mulf3(dir, sc.bounce_offset)); out.d = dir; out.dist = remaining;
        float dp = max_ref(0.0f, dot3(h.nrm, dir));
        r.att = mulf3(rgb, dp);
        if (m.type == RT_MAT_CHECKER) r.att = mulf3(r.att, factor);
    }
    else if (m.type == RT_MAT_REFLECTIVE)
    {
        if (preview) { r.att = rgb; return r; }
        float remaining = in.dist - h.dist;
        float3 nd = reflect3(in.d, h.nrm);
        if (m.scalar > 0.0f)
        {
            nd = add3(nd, mulf3(random_unit_vector(rng), m.scalar));
            nd = normalized3(nd);
        }
        out.o = add3(h.pos, mulf3(nd, sc.bounce_offset)); out.d = nd; out.dist = remaining;
        r.att = rgb;
    }
    else if (m.type == RT_MAT_EMISSIVE)
    {
        if (preview) { r.att = rgb; return r; }
        out = in;
        r.emi = rgb;
    }
    else if (m.type == RT_MAT_NULL)
    {
        if (preview) return r;
        float remaining = in.dist - h.dist;
        out.o = add3(h.pos, mulf3(in.d, sc.bounce_offset)); out.d = in.d; out.dist = remaining;
        r.att = V3(1, 1, 1);
    }
    return r;
}

// ISurfaceMaterial::BounceViewRay / PreviewColor over a material tree.  Blend draws one Random()
// and evaluates one child (SurfaceMaterials.cpp:153-161).  Combine evaluates B, then A — the
// order the compiled reference uses for `A->Bounce(..) + B->Bounce(..)` (:169-177; pinned by
// tests/test_oracle_vs_ref.py) — so the outgoing ray and the later RNG draws are A's.
static __device__ __noinline__ Bounce material_eval(const DevScene& sc, int root, bool preview,
                                             const Ray& in, const Hit& h, Ray& out, Rng& rng)
{
    int frame_node[RT_MAX_MATERIAL_DEPTH];
    Bounce frame_b[RT_MAX_MATERIAL_DEPTH];
    bool frame_second[RT_MAX_MATERIAL_DEPTH];
    int top = 0;
    int node = root;
    Bounce r;
    for (;;)
    {
        // descend to a leaf
        r.att = V3(0, 0, 0); r.emi = V3(0, 0, 0);
        while (node >= 0)
        {
            const rt_material m = sc.materials[node];
            if (m.type == RT_MAT_BLEND)
            {
                node = rng_random(rng) > m.scalar ? m.child_a : m.child_b;
                continue;
            }
            if (m.type == RT_MAT_COMBINE && top < RT_MAX_MATERIAL_DEPTH)
            {
                frame_node[top] = node; frame_second[top] = false; top++;
                node = m.child_b;
                continue;
            }
            r = material_leaf(sc, m, preview, in, h, out, rng);
            break;
        }
        // ascend through finished Combine frames
        bool descend = false;
        while (top > 0)
        {
            if (!frame_second[top - 1])
            {
                frame_b[top - 1] = r;
                frame_second[top - 1] = true;
                node = sc.materials[frame_node[top - 1]].child_a;
                descend = true;
                break;
            }
            const Bounce b = frame_b[top - 1];
            r.att = add3(r.att, b.att);       // A + B
            r.emi = add3(r.emi, b.emi);
            top--;
        }
        if (!descend) return r;
    }
}

__device__ __forceinline__ bool is_non_zero(float3 a) { return !eq_zero(a.x) && !eq_zero(a.y) && !eq_zero(a.z); }   // RVector.h:142-145

__device__ __forceinline__ float3 sky_color(float3 d)                       // RayTracerScene.cpp:92-93
{
    float t = 0.5f * (d.y + 1.0f);
    return add3(mulf3(V3(1.0f, 1.0f, 1.0f), 1.0f - t), mulf3(V3(0.5f, 0.7f, 1.0f), t));
}

// LinearToGamma + MakePixelColor, ColorBuffer.h:81-109 (non-OSX ARGB packing).  powf is CUDA's:
// the 8-bit result may differ from glibc's by one code value at a rounding boundary.
__device__ __forceinline__ uint32_t make_pixel(float3 lin)
{
    const float e = 1.0f / 2.2f;
    float3 g = V3(powf(lin.x, e), powf(lin.y, e), powf(lin.z, e));
    int r = (int)(min_ref(max_ref(g.x, 0.0f), 1.0f) * 255);
    int gg = (int)(min_ref(max_ref(g.y, 0.0f), 1.0f) * 255);
    int b = (int)(min_ref(max_ref(g.z, 0.0f), 1.0f) * 255);
    return (255u << 24) | ((uint32_t)(r & 255) << 16) | ((uint32_t)(gg & 255) << 8) | (uint32_t)(b & 255);
}

// ---- camera -----------------------------------------------------------------------------------------
// ThreadWorker_Render's ray generator (RayTracerProgram.cpp:133-165) with W,H as parameters;
// sub < 0: one un-jittered ray through the pixel's base direction; sub 0..3: the
// ENABLE_ANTIALIASING sub-sample with two Random() draws of jitter (:146-165).
// the pixel's base direction (dx, dy): the part of the generator that does not depend on the sample
__device__ __forceinline__ void camera_base(int width, int height, int x, int y, float& dx, float& dy)
{
    // x = pixel % width, y = pixel / width                               // ColorBuffer.h:19-23
    const float aspect = (float)width / (float)height;
    dx = -(float)(x - width / 2) / (float)(width * 2) * aspect;
    dy = -(float)(y - height / 2) / (float)(height * 2);
}

__device__ __forceinline__ Ray camera_ray_from_base(const DevScene& sc, int width, float dx, float dy, int sub, Rng& rng)
{
    float ox = 0.0f, oy = 0.0f;
    if (sub >= 0)
    {
        const float inv_pixel_radius = 1.0f / (float)(width * 4);
        const float offset_radius = inv_pixel_radius * 0.5f;
        ox = (sub & 1) ? inv_pixel_radius : 0.0f;
        oy = (sub & 2) ? inv_pixel_radius : 0.0f;
        ox += (rng_random(rng) - 0.5f) * offset_radius;
        oy += (rng_random(rng) - 0.5f) * offset_radius;
    }
    Ray r;
    r.o = V3(sc.eye[0], sc.eye[1], sc.eye[2]);
    r.d = normalized3(V3(dx + ox, dy + oy, sc.dir_z));
    r.dist = sc.ray_distance;
    return r;
}

__device__ __forceinline__ Ray camera_ray(const DevScene& sc, int width, int height, int x, int y, int sub, Rng& rng)
{
    float dx, dy;
    camera_base(width, height, x, y, dx, dy);
    return camera_ray_from_base(sc, width, dx, dy, sub, rng);
}

} // namespace rtdev
