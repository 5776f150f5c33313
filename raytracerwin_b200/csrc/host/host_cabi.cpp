// host_cabi.cpp — extern "C" handles over the C++ scene layer (include/rt_host.h).
#include "rt_host.h"
#include "rt_host.hpp"

#include <string.h>
#include <stdlib.h>

using namespace rtb200;

struct rt_host_scene { RayTracerProgram program; };
struct rt_host_material { std::unique_ptr<ISurfaceMaterial> m; };

static thread_local std::string g_error;

static std::unique_ptr<ISurfaceMaterial> take(rt_host_material* h)
{
    if (!h) return nullptr;
    std::unique_ptr<ISurfaceMaterial> m = std::move(h->m);
    delete h;
    return m;
}

// No C++ exception crosses the C ABI (include/rt_host.h): entries report RT_ERR_NOMEM / RT_ERR_INVALID
// (or null) and leave the message in rt_host_last_error().
static void note_error(const char* what) noexcept
{
    try { g_error = what; } catch (...) {}
}

template <typename F>
static int guard(F&& f) noexcept
{
    try { return f(); }
    catch (const std::bad_alloc&) { note_error("out of host memory"); return RT_ERR_NOMEM; }
    catch (const std::exception& e) { note_error(e.what()); return RT_ERR_INVALID; }
    catch (...) { note_error("unexpected C++ exception"); return RT_ERR_INVALID; }
}

template <typename T, typename F>
static T* guard_ptr(F&& f) noexcept
{
    try { return f(); }
    catch (const std::bad_alloc&) { note_error("out of host memory"); }
    catch (const std::exception& e) { note_error(e.what()); }
    catch (...) { note_error("unexpected C++ exception"); }
    return nullptr;
}

template <typename M, typename... A>
static rt_host_material* make(A&&... a) noexcept
{
    return guard_ptr<rt_host_material>([&]() {
        std::unique_ptr<rt_host_material> h(new rt_host_material());
        h->m.reset(new M(std::forward<A>(a)...));
        return h.release();
    });
}

extern "C" {

const char* rt_host_last_error(void) { return g_error.c_str(); }

rt_host_scene* rt_host_scene_new(void) { return guard_ptr<rt_host_scene>([]() { return new rt_host_scene(); }); }
void rt_host_scene_free(rt_host_scene* s) { delete s; }

rt_host_material* rt_host_mat_diffuse(float r, float g, float b) { return make<SurfaceMaterial_Diffuse>(RVec3(r, g, b)); }
rt_host_material* rt_host_mat_checker(float r, float g, float b, float size) { return make<SurfaceMaterial_DiffuseChecker>(RVec3(r, g, b), size); }
rt_host_material* rt_host_mat_reflective(float r, float g, float b, float fuzz) { return make<SurfaceMaterial_Reflective>(RVec3(r, g, b), fuzz); }
rt_host_material* rt_host_mat_emissive(float r, float g, float b) { return make<SurfaceMaterial_Emissive>(RVec3(r, g, b)); }
rt_host_material* rt_host_mat_null(void) { return make<SurfaceMaterial_Null>(); }
rt_host_material* rt_host_mat_blend(rt_host_material* a, rt_host_material* b, float f) { return make<SurfaceMaterial_Blend>(take(a), take(b), f); }
rt_host_material* rt_host_mat_combine(rt_host_material* a, rt_host_material* b) { return make<SurfaceMaterial_Combine>(take(a), take(b)); }

static int add(rt_host_scene* s, std::unique_ptr<RShape> shape, rt_host_material* mat)
{
    if (!s) { g_error = "null scene"; return RT_ERR_INVALID; }
    RayTracerScene* scene = s->program.GetScene();
    scene->AddShape(std::move(shape), take(mat));
    return scene->NumShapes() - 1;
}

int rt_host_add_sphere(rt_host_scene* s, const float c[3], float r, rt_host_material* mat)
{
    return add(s, RSphere::Create(RVec3(c), r), mat);
}
int rt_host_add_plane(rt_host_scene* s, const float n[3], const float p[3], rt_host_material* mat)
{
    return add(s, RPlane::Create(RVec3(n), RVec3(p)), mat);
}
int rt_host_add_capsule(rt_host_scene* s, const float a[3], const float b[3], float r, rt_host_material* mat)
{
    return add(s, RCapsule::Create(RVec3(a), RVec3(b), r), mat);
}
int rt_host_add_triangle(rt_host_scene* s, const float p[9], rt_host_material* mat)
{
    return add(s, RTriangle::Create(RVec3(p), RVec3(p + 3), RVec3(p + 6)), mat);
}
int rt_host_add_mesh_obj(rt_host_scene* s, const char* path, rt_host_material* mat)
{
    return guard([&]() -> int {
        std::unique_ptr<RMeshShape> m = RMeshShape::Create(path);
        if (!m->IsLoaded())
        {
            g_error = m->Error();
            take(mat);
            return RT_ERR_INVALID;
        }
        return add(s, std::move(m), mat);
    });
}
int rt_host_add_mesh_arrays(rt_host_scene* s, const float* points, int num_points,
                            const float* normals, int num_normals, const float* texcoords, int num_texcoords,
                            const int32_t* pidx, const int32_t* nidx, const int32_t* tidx, int num_tris,
                            rt_host_material* mat)
{
    return guard([&]() -> int {
        if (!points || !pidx || num_points <= 0 || num_tris <= 0) { g_error = "empty mesh"; take(mat); return RT_ERR_INVALID; }
        std::unique_ptr<RMeshShape> m(new RMeshShape(points, num_points, normals, num_normals, texcoords, num_texcoords, pidx, nidx, tidx, num_tris));
        if (!m->IsLoaded())
        {
            g_error = m->Error();
            take(mat);
            return RT_ERR_INVALID;
        }
        return add(s, std::move(m), mat);
    });
}

int rt_host_setup_default_scene(rt_host_scene* s, const char* data_dir)
{
    return guard([&]() -> int {
        if (!s) return RT_ERR_INVALID;
        s->program.SetupScene(data_dir ? data_dir : "Data");
        RayTracerScene* scene = s->program.GetScene();
        RMeshShape* mesh = scene->GetShape(scene->NumShapes() - 1)->AsMesh();
        if (!mesh || !mesh->IsLoaded()) { g_error = mesh ? mesh->Error() : "no mesh"; return RT_ERR_INVALID; }
        return RT_OK;
    });
}

int rt_host_use_device_bvh_builder(rt_gpu_ctx* ctx)
{
    return guard([&]() -> int {
        SetDeviceBvhBuilder(ctx);
        return RT_OK;
    });
}

int rt_host_clear_lights(rt_host_scene* s) { s->program.GetScene()->Lights.clear(); return RT_OK; }
int rt_host_add_light(rt_host_scene* s, int type, const float v[3], const float color[3])
{
    return guard([&]() -> int {
        LightData l; l.Type = type; l.PositionOrDirection = RVec3(v); l.Color = RVec3(color);
        s->program.GetScene()->Lights.push_back(l);
        return RT_OK;
    });
}

int rt_host_set_unit_vectors(rt_host_scene* s, uint32_t seed, uint32_t count)
{
    return guard([&]() -> int {
        s->program.GetScene()->SetUnitVectors(seed, count);
        return RT_OK;
    });
}

const rt_scene_desc* rt_host_scene_desc(rt_host_scene* s)
{
    return guard_ptr<const rt_scene_desc>([&]() { return &s->program.GetScene()->Flatten(); });
}

static RMeshShape* mesh_of(rt_host_scene* s, int shape)
{
    RayTracerScene* scene = s->program.GetScene();
    if (shape < 0 || shape >= scene->NumShapes()) return nullptr;
    return scene->GetShape(shape)->AsMesh();
}

int rt_host_mesh_counts(rt_host_scene* s, int shape, int32_t out[7])
{
    return guard([&]() -> int {
        RMeshShape* m = mesh_of(s, shape);
        if (!m) return RT_ERR_INVALID;
        out[0] = (int)m->Points.size(); out[1] = (int)m->Texcoords.size(); out[2] = (int)m->Normals.size();
        out[3] = (int)m->PointIndices.size() / 3; out[4] = (int)m->Textures.size();
        out[5] = (int)m->GetFlat().nodes.size(); out[6] = m->GetFlat().depth;
        return RT_OK;
    });
}

int rt_host_mesh_dump(rt_host_scene* s, int shape, float* points, float* texcoords, float* normals,
                      int32_t* pidx, int32_t* tidx, int32_t* nidx, int32_t* matid)
{
    return guard([&]() -> int {
        RMeshShape* m = mesh_of(s, shape);
        if (!m) return RT_ERR_INVALID;
        memcpy(points, m->Points.data(), m->Points.size() * sizeof(RVec3));
        memcpy(texcoords, m->Texcoords.data(), m->Texcoords.size() * sizeof(RVec3));
        memcpy(normals, m->Normals.data(), m->Normals.size() * sizeof(RVec3));
        memcpy(pidx, m->PointIndices.data(), m->PointIndices.size() * sizeof(int));
        memcpy(tidx, m->TexcoordIndices.data(), m->TexcoordIndices.size() * sizeof(int));
        memcpy(nidx, m->NormalIndices.data(), m->NormalIndices.size() * sizeof(int));
        memcpy(matid, m->PolyMaterialId.data(), m->PolyMaterialId.size() * sizeof(int));
        return RT_OK;
    });
}

int rt_host_mesh_texture_info(rt_host_scene* s, int shape, int slot, int32_t wh[2])
{
    return guard([&]() -> int {
        RMeshShape* m = mesh_of(s, shape);
        if (!m || slot < 0 || slot >= (int)m->Textures.size()) return RT_ERR_INVALID;
        wh[0] = m->Textures[slot] ? m->Textures[slot]->Width : 0;
        wh[1] = m->Textures[slot] ? m->Textures[slot]->Height : 0;
        return RT_OK;
    });
}

int rt_host_mesh_texture_pixels(rt_host_scene* s, int shape, int slot, float* out)
{
    return guard([&]() -> int {
        RMeshShape* m = mesh_of(s, shape);
        if (!m || slot < 0 || slot >= (int)m->Textures.size() || !m->Textures[slot]) return RT_ERR_INVALID;
        m->Textures[slot]->ExpandTo(out);
        return RT_OK;
    });
}

int rt_host_texel_lut(float* out512)
{
    if (!out512) { g_error = "rt_host_texel_lut: out512 is null"; return RT_ERR_INVALID; }
    RTexture::MakeLut(out512);
    return RT_OK;
}

int rt_host_decode_png(const char* path, int32_t wh[2], int32_t* channels, uint8_t** out_pixels)
{
    return guard([&]() -> int {
        int w, h, ch;
        std::vector<uint8_t> px;
        std::string err;
        if (!DecodePng8(path, w, h, ch, px, err)) { g_error = err; return RT_ERR_INVALID; }
        wh[0] = w; wh[1] = h; *channels = ch;
        *out_pixels = (uint8_t*)malloc(px.size());
        if (!*out_pixels) return RT_ERR_NOMEM;
        memcpy(*out_pixels, px.data(), px.size());
        return RT_OK;
    });
}

void rt_host_free(void* p) { free(p); }

int rt_host_write_png_argb(const char* path, const uint32_t* argb, int32_t width, int32_t height)
{
    return guard([&]() -> int { return WritePngARGB(path, argb, width, height) ? RT_OK : RT_ERR_INVALID; });
}

int rt_host_program_run(rt_host_scene* s, int device, int32_t width, int32_t height, int32_t passes,
                        int32_t max_bounce, uint32_t seed, const char* png_path, double* out_seconds, uint64_t* out_rays)
{
    return guard([&]() -> int {
        std::string err;
        int rc = s->program.Run(device, width, height, passes, max_bounce, seed, png_path ? png_path : "", out_seconds, out_rays, &err);
        if (rc != RT_OK) g_error = err;
        return rc;
    });
}

} // extern "C"
