// rt_host.hpp — host-side (CPU) scene layer of the B200 path.
//
// Same public surface as the reference for everything that BUILDS a scene
// (RayTracerScene.h:43-62, Shapes.h:17-123, MeshShape.h:16-38, SurfaceMaterials.h:35-141,
// RayTracerProgram.h:25-62); nothing here traces rays.  Where the reference's classes carry
// virtual TestRayIntersection / BounceViewRay methods that run per ray on the CPU, these
// classes carry a Flatten() that emits plain-old-data for the device instead: the per-ray work
// lives in csrc/rt_wave_kernels.cuh + rt_device.cuh (launched from csrc/rt_gpu.cu) behind include/rt_gpu.h.
#pragma once

#include <memory>
#include <string>
#include <vector>
#include <stdint.h>

#include "rt_gpu.h"

namespace rtb200 {

struct RVec3
{
    float x, y, z;
    RVec3() : x(0.0f), y(0.0f), z(0.0f) {}
    RVec3(float _x, float _y, float _z) : x(_x), y(_y), z(_z) {}
    explicit RVec3(const float* v) : x(v[0]), y(v[1]), z(v[2]) {}
};

struct RAabb
{
    RVec3 pMin, pMax;
    RAabb();                                   // empty box (+FLT_MAX / -FLT_MAX), RAabb.cpp:12-16
    void Expand(const RVec3& p);
    void ExpandBySphere(const RVec3& c, float r);
};

struct RenderOption { bool UseBaseColor = false; };   // RayTracerScene.h:27-35

// ---- materials ---------------------------------------------------------------------------
class ISurfaceMaterial
{
public:
    virtual ~ISurfaceMaterial() {}
    // Appends this subtree to `out` (children first) and returns the index of its root node.
    virtual int Flatten(std::vector<rt_material>& out) const = 0;
};

class SurfaceMaterial_Diffuse : public ISurfaceMaterial
{
public:
    explicit SurfaceMaterial_Diffuse(const RVec3& InAlbedo = RVec3(1.0f, 1.0f, 1.0f)) : Albedo(InAlbedo) {}
    int Flatten(std::vector<rt_material>& out) const override;
protected:
    RVec3 Albedo;
};

class SurfaceMaterial_DiffuseChecker : public SurfaceMaterial_Diffuse
{
public:
    explicit SurfaceMaterial_DiffuseChecker(const RVec3& InAlbedo = RVec3(1.0f, 1.0f, 1.0f), float InPatternSize = 5.0f);
    int Flatten(std::vector<rt_material>& out) const override;
private:
    float ReciprocalPatternSize;
};

class SurfaceMaterial_Reflective : public ISurfaceMaterial
{
public:
    explicit SurfaceMaterial_Reflective(const RVec3& InAlbedo = RVec3(1.0f, 1.0f, 1.0f), float InFuzziness = 0.0f)
        : Albedo(InAlbedo), Fuzziness(InFuzziness) {}
    int Flatten(std::vector<rt_material>& out) const override;
private:
    RVec3 Albedo;
    float Fuzziness;
};

class SurfaceMaterial_Emissive : public ISurfaceMaterial
{
public:
    explicit SurfaceMaterial_Emissive(const RVec3& InColor) : Color(InColor) {}
    int Flatten(std::vector<rt_material>& out) const override;
private:
    RVec3 Color;
};

class SurfaceMaterial_Blend : public ISurfaceMaterial
{
public:
    SurfaceMaterial_Blend(std::unique_ptr<ISurfaceMaterial> InMaterialA, std::unique_ptr<ISurfaceMaterial> InMaterialB, float InBlendFactor);
    int Flatten(std::vector<rt_material>& out) const override;
private:
    std::unique_ptr<ISurfaceMaterial> BlendMaterialA, BlendMaterialB;
    float BlendFactor;
};

class SurfaceMaterial_Combine : public ISurfaceMaterial
{
public:
    SurfaceMaterial_Combine(std::unique_ptr<ISurfaceMaterial> InMaterialA, std::unique_ptr<ISurfaceMaterial> InMaterialB)
        : MaterialA(std::move(InMaterialA)), MaterialB(std::move(InMaterialB)) {}
    int Flatten(std::vector<rt_material>& out) const override;
private:
    std::unique_ptr<ISurfaceMaterial> MaterialA, MaterialB;
};

class SurfaceMaterial_Null : public ISurfaceMaterial
{
public:
    int Flatten(std::vector<rt_material>& out) const override;
};

// ---- shapes --------------------------------------------------------------------------------
class RMeshShape;

class RShape
{
public:
    virtual ~RShape() {}
    void SetSurfaceMaterial(std::unique_ptr<ISurfaceMaterial> InMaterial) { SurfaceMaterial = std::move(InMaterial); }
    ISurfaceMaterial* GetSurfaceMaterial() { return SurfaceMaterial.get(); }
    virtual bool HasCullingBounds() const { return true; }
    const RAabb& GetBounds() const { return Aabb; }
    // Fills type/params/bounds of the POD record (material and mesh indices are set by the scene).
    virtual void Flatten(rt_shape& out) const = 0;
    virtual RMeshShape* AsMesh() { return nullptr; }
protected:
    void FlattenCommon(rt_shape& out, int type) const;
    RAabb Aabb;
    std::unique_ptr<ISurfaceMaterial> SurfaceMaterial;
};

class RSphere : public RShape
{
public:
    RVec3 Center; float Radius;
    RSphere(const RVec3& InCenter, float InRadius);
    static std::unique_ptr<RSphere> Create(const RVec3& c, float r) { return std::unique_ptr<RSphere>(new RSphere(c, r)); }
    void Flatten(rt_shape& out) const override;
};

class RPlane : public RShape
{
public:
    RVec3 Normal, Point;
    RPlane(const RVec3& InNormal, const RVec3& InPoint) : Normal(InNormal), Point(InPoint) {}
    static std::unique_ptr<RShape> Create(const RVec3& n, const RVec3& p) { return std::unique_ptr<RShape>(new RPlane(n, p)); }
    bool HasCullingBounds() const override { return false; }      // infinite, never culled
    void Flatten(rt_shape& out) const override;
};

class RCapsule : public RShape
{
public:
    RVec3 Start, End; float Radius;
    RCapsule(const RVec3& InStart, const RVec3& InEnd, float InRadius);
    static std::unique_ptr<RShape> Create(const RVec3& a, const RVec3& b, float r) { return std::unique_ptr<RShape>(new RCapsule(a, b, r)); }
    void Flatten(rt_shape& out) const override;
};

class RTriangle : public RShape
{
public:
    RVec3 Points[3];
    RTriangle(const RVec3& p0, const RVec3& p1, const RVec3& p2);
    static std::unique_ptr<RShape> Create(const RVec3& p0, const RVec3& p1, const RVec3& p2) { return std::unique_ptr<RShape>(new RTriangle(p0, p1, p2)); }
    void Flatten(rt_shape& out) const override;
};

// Decoded texture.  The reference keeps RVec4 texels, rgb linearised with powf(c / 255, 2.2f) per texel
// (Texture.cpp:119-151); powf only ever sees 256 inputs there, so this class keeps the PNG's 8-bit texels and the
// 512-entry table (rgb | alpha) instead — the device expands them (rt_texture in rt_gpu.h), ExpandTo() does it on
// the host for whoever wants the float texels; both give the reference's bits.
struct RTexture
{
    int Width = 0, Height = 0, Channels = 0;
    std::vector<uint8_t> Pixels8;  // Channels * Width * Height
    float Lut[512];                // [c] = powf(c / 255, 2.2f), [256 + c] = c / 255
    void ExpandTo(float* OutRGBA) const;     // 4 * Width * Height floats
    static std::unique_ptr<RTexture> LoadTexturePNG(const std::string& Filename);
    static void MakeLut(float* Out512);      // the table above (rt_host_texel_lut hands it to callers)
};

// Pre-order flattened BVH of one mesh + device-ready triangle/shading records.
struct FlatMesh
{
    std::vector<rt_bvh_node> nodes;
    std::vector<rt_tri> tris;       // leaf order
    std::vector<rt_shade> shade;    // original order
    std::vector<rt_texture> textures;
    int depth = 0;
};

class RMeshShape : public RShape
{
public:
    explicit RMeshShape(const std::string& Filename);            // OBJ (+MTL, +PNG) from disk
    RMeshShape(const float* points, int num_points, const float* normals, int num_normals,
               const float* texcoords, int num_texcoords, const int32_t* pidx, const int32_t* nidx,
               const int32_t* tidx, int num_tris);
    static std::unique_ptr<RMeshShape> Create(const std::string& Filename) { return std::unique_ptr<RMeshShape>(new RMeshShape(Filename)); }

    void Flatten(rt_shape& out) const override;
    RMeshShape* AsMesh() override { return this; }
    bool IsLoaded() const { return Loaded; }
    const std::string& Error() const { return ErrorText; }
    const FlatMesh& GetFlat() const { return Flat; }

    // raw arrays, named as in MeshShape.h:24-37
    std::vector<RVec3> Points, Texcoords, Normals;
    std::vector<int> PointIndices, TexcoordIndices, NormalIndices;
    std::vector<int> PolyMaterialId;
    std::vector<std::unique_ptr<RTexture>> Textures;   // indexed by material id

private:
    void BuildSpatial();         // KdTree::Build equivalent + flattening
    bool Loaded = false;
    bool BuildFailed = false;
    std::string ErrorText;
    FlatMesh Flat;
};

// Where meshes get their tree: the host builder below, or (opt-in, SetDeviceBvhBuilder) rt_gpu_build_bvh on the
// given context — same arrays bit for bit, ~25x faster at 10 M triangles.  nullptr switches back to the host.
void SetDeviceBvhBuilder(rt_gpu_ctx* ctx);

// Builds the reference's tree (KdTree.cpp:37-126) directly in pre-order.  Returns the depth.
int BuildFlatBvh(const RVec3* Points, const int* Indices, int NumTriangles,
                 std::vector<rt_bvh_node>& nodes, std::vector<rt_tri>& tris);

// ---- scene ---------------------------------------------------------------------------------
struct LightData { int Type; RVec3 PositionOrDirection; RVec3 Color; };   // Light.h:16-21

class RayTracerScene
{
public:
    RayTracerScene();
    // Add a shape to scene (RayTracerScene.cpp:25-29)
    void AddShape(std::unique_ptr<RShape> Shape, std::unique_ptr<ISurfaceMaterial> SurfaceMaterial);
    int NumShapes() const { return (int)SceneShapes.size(); }
    RShape* GetShape(int i) { return SceneShapes[i].get(); }

    std::vector<LightData> Lights;                 // defaults to GSceneLights
    void SetUnitVectors(uint32_t seed, uint32_t count);

    // POD view for rt_gpu_upload_scene; rebuilt lazily after AddShape.
    const rt_scene_desc& Flatten();

private:
    std::vector<std::unique_ptr<RShape>> SceneShapes;
    bool Dirty = true;
    rt_scene_desc Desc;
    std::vector<rt_shape> FlatShapes;
    std::vector<rt_material> FlatMaterials;
    std::vector<rt_mesh> FlatMeshes;
    std::vector<rt_light> FlatLights;
    std::vector<float> UnitVectors;
};

// PseudoRandomUnitVectors (Math.cpp:24-31) from the counter RNG; multi-threaded.
void GenerateUnitVectors(uint32_t seed, uint32_t count, float* out_xyz);

// Headless program shell: preview pass + N accumulation passes on one GPU.
class RayTracerProgram
{
public:
    RayTracerProgram() {}
    RayTracerScene* GetScene() { return &Scene; }
    void SetupScene(const std::string& DataDir);   // the reference's default scene
    // returns 0 on success; fills seconds and ray count of the accumulation passes
    int Run(int Device, int Width, int Height, int Passes, int MaxBounceTimes, uint32_t Seed,
            const std::string& PngPath, double* OutSeconds, uint64_t* OutRays, std::string* Error);
private:
    RayTracerScene Scene;
};

bool WritePngARGB(const std::string& Filename, const uint32_t* Pixels, int Width, int Height);
bool DecodePng8(const std::string& Filename, int& Width, int& Height, int& Channels,
                std::vector<uint8_t>& Pixels, std::string& Error);

} // namespace rtb200
