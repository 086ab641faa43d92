// host_capi.cpp — C entry points over the C++ host (RenderGraph + HybridRenderPath) for harnesses that are not C++
// (tests, bench.py). A C++ maintainer of the reference uses the classes directly; see INTEGRATION.md.
#include <string.h>

#include <memory>

#include "hybrid_render_path.h"
#include "raytraced_render_path.h"
#include "scene_loader.h"

struct vhrh_renderer {
    std::unique_ptr<ResourceManager> resource_manager;
    std::unique_ptr<RenderGraph> render_graph;
    std::unique_ptr<HybridRenderPath> path;
    std::unique_ptr<RaytracedRenderPath> raytraced_path;
    RenderPath *active = nullptr;          // the path whose nodes are registered (Renderer::active_render_path, renderer.h)
    std::string error;
    bool built = false;
};

namespace {
thread_local std::string g_host_error;
template <typename F>
int guarded(vhrh_renderer *r, F &&f) {
    try {
        f();
        return VHR_OK;
    } catch (const VhrHostError &e) {
        g_host_error = e.message;
        if (r) r->error = e.message;
        return e.status;
    } catch (const std::exception &e) {
        g_host_error = e.what();
        return VHR_ERR_INVALID;
    }
}
}  // namespace

extern "C" {

const char *vhrh_last_error(void) { return g_host_error.c_str(); }

// Renderer::Renderer (renderer.cpp:18-44) minus window / swapchain / UI
int vhrh_renderer_create(int device, void *cuda_stream, uint32_t width, uint32_t height, vhrh_renderer **out) {
    if (!out) return VHR_ERR_INVALID;
    *out = nullptr;
    auto r = std::make_unique<vhrh_renderer>();
    int rc = guarded(r.get(), [&] {
        r->resource_manager = std::make_unique<ResourceManager>(device, cuda_stream, width, height);
        r->render_graph = std::make_unique<RenderGraph>(*r->resource_manager);
        r->path = std::make_unique<HybridRenderPath>(*r->render_graph, *r->resource_manager);
        r->raytraced_path = std::make_unique<RaytracedRenderPath>(*r->render_graph, *r->resource_manager);
    });
    if (rc == VHR_OK) *out = r.release();
    return rc;
}

void vhrh_renderer_destroy(vhrh_renderer *r) {
    if (!r) return;
    guarded(r, [&] {
        if (r->built && r->active) r->active->DeregisterPath(*r->render_graph, *r->resource_manager);
    });
    delete r;
}

vhr_context *vhrh_context(vhrh_renderer *r) { return r ? r->resource_manager->ctx : nullptr; }

// SceneLoader::LoadScene -> ResourceManager::UpdateGeometry (scene_loader.cpp:331): flat arrays, one mesh per
// `prims_per_mesh` primitives (0 = a single mesh); the flat primitive order is what matters (object ids).
int vhrh_load_scene(vhrh_renderer *r, const void *vertices, uint32_t n_vertices, const uint32_t *indices, uint32_t n_indices,
                    const void *primitives, uint32_t n_primitives, uint32_t prims_per_mesh) {
    if (!r) return VHR_ERR_INVALID;
    return guarded(r, [&] {
        std::vector<Vertex> v((const Vertex *)vertices, (const Vertex *)vertices + n_vertices);
        std::vector<uint32_t> idx(indices, indices + n_indices);
        Scene scene;
        const Primitive *p = (const Primitive *)primitives;
        uint32_t per = prims_per_mesh ? prims_per_mesh : (n_primitives ? n_primitives : 1);
        for (uint32_t i = 0; i < n_primitives; i += per) {
            Mesh m;
            for (uint32_t k = i; k < n_primitives && k < i + per; ++k) m.primitives.push_back(p[k]);
            scene.meshes.push_back(std::move(m));
        }
        r->resource_manager->UpdateGeometry(v, idx, scene);
    });
}

// ---- glTF scene path (scene_loader.h) ----------------------------------------------------------------------------------
struct vhrh_parsed_scene { SceneLoader::ParsedScene parsed; };

// SceneLoader::ParseScene: file -> flat arrays, no GPU involved
int vhrh_parse_gltf(const char *path, vhrh_parsed_scene **out) {
    if (!path || !out) return VHR_ERR_INVALID;
    *out = nullptr;
    auto p = std::make_unique<vhrh_parsed_scene>();
    int rc = guarded(nullptr, [&] { SceneLoader::ParseScene(path, p->parsed); });
    if (rc == VHR_OK) *out = p.release();
    return rc;
}
void vhrh_parsed_scene_destroy(vhrh_parsed_scene *p) { delete p; }
// counts[5] = vertices, indices, primitives, textures, meshes
int vhrh_parsed_scene_counts(vhrh_parsed_scene *p, uint32_t *counts) {
    if (!p || !counts) return VHR_ERR_INVALID;
    uint32_t prims = 0;
    for (const Mesh &m : p->parsed.scene.meshes) prims += (uint32_t)m.primitives.size();
    counts[0] = (uint32_t)p->parsed.vertices.size(); counts[1] = (uint32_t)p->parsed.indices.size(); counts[2] = prims;
    counts[3] = (uint32_t)p->parsed.textures.size(); counts[4] = (uint32_t)p->parsed.scene.meshes.size();
    return VHR_OK;
}
// copies the flat arrays out (buffers sized from vhrh_parsed_scene_counts); primitives in mesh order = object ids
int vhrh_parsed_scene_copy(vhrh_parsed_scene *p, void *vertices, uint32_t *indices, void *primitives, uint32_t *prims_per_mesh, void *camera,
                           void *directional_light) {
    if (!p) return VHR_ERR_INVALID;
    const SceneLoader::ParsedScene &s = p->parsed;
    if (vertices && !s.vertices.empty()) memcpy(vertices, s.vertices.data(), s.vertices.size() * sizeof(Vertex));
    if (indices && !s.indices.empty()) memcpy(indices, s.indices.data(), s.indices.size() * sizeof(uint32_t));
    Primitive *out = (Primitive *)primitives;
    size_t k = 0, mi = 0;
    for (const Mesh &m : s.scene.meshes) {
        if (prims_per_mesh) prims_per_mesh[mi] = (uint32_t)m.primitives.size();
        ++mi;
        for (const Primitive &pr : m.primitives) { if (out) out[k] = pr; ++k; }
    }
    if (camera) memcpy(camera, &s.scene.camera, sizeof(Camera));
    if (directional_light) memcpy(directional_light, &s.scene.directional_light, sizeof(DirectionalLight));
    return VHR_OK;
}
// info[7] = width, height, VkFormat, mag, min, address u, address v; rgba may be NULL
int vhrh_parsed_scene_texture(vhrh_parsed_scene *p, uint32_t index, int32_t *info, uint8_t *rgba) {
    if (!p || index >= p->parsed.textures.size() || !info) return VHR_ERR_INVALID;
    const SceneLoader::ParsedTexture &t = p->parsed.textures[index];
    info[0] = (int32_t)t.width; info[1] = (int32_t)t.height; info[2] = (int32_t)t.format;
    info[3] = t.sampler.mag_filter; info[4] = t.sampler.min_filter; info[5] = t.sampler.address_mode_u; info[6] = t.sampler.address_mode_v;
    if (rgba) memcpy(rgba, t.rgba.data(), t.rgba.size());
    return VHR_OK;
}
// SceneLoader::LoadScene (scene_loader.cpp:336-349) on the renderer's ResourceManager: textures, then UpdateGeometry.
// An unreadable file leaves an empty scene, like the reference; returns the number of primitives loaded.
int vhrh_load_gltf(vhrh_renderer *r, const char *path) {
    if (!r || !path) return VHR_ERR_INVALID;
    int n = 0;
    int rc = guarded(r, [&] {
        Scene s = SceneLoader::LoadScene(*r->resource_manager, path);
        for (const Mesh &m : s.meshes) n += (int)m.primitives.size();
    });
    return rc == VHR_OK ? n : rc;
}
// wh[2] receives the extent; rgba (capacity bytes) the RGBA8 texels when large enough
int vhrh_has_stb_image(void) { return SceneLoader::HasStbImage() ? 1 : 0; }
int vhrh_has_cgltf(void) { return SceneLoader::HasCgltf() ? 1 : 0; }

int vhrh_decode_png(const uint8_t *data, size_t size, uint32_t *wh, uint8_t *rgba, size_t capacity) {
    if (!data || !wh) return VHR_ERR_INVALID;
    std::vector<uint8_t> out;
    std::string err;
    if (!SceneLoader::DecodePNG(data, size, wh[0], wh[1], out, err)) { g_host_error = err; return VHR_ERR_INVALID; }
    if (rgba && capacity >= out.size()) memcpy(rgba, out.data(), out.size());
    return VHR_OK;
}

// The ImGui radio buttons of HybridRenderPath::ImGuiDrawSettings (hybrid_render_path.cpp:394-441) + Rebuild().
int vhrh_set_modes(vhrh_renderer *r, int shadow_mode, int ambient_occlusion_mode, int reflection_mode, int denoise, int svgf_fused) {
    if (!r) return VHR_ERR_INVALID;
    return guarded(r, [&] {
        r->path->shadow_mode = shadow_mode;
        r->path->ambient_occlusion_mode = ambient_occlusion_mode;
        r->path->reflection_mode = reflection_mode;
        r->path->denoise_shadow_and_ao = denoise != 0;
        r->path->svgf_fused = svgf_fused != 0;
        if (r->built && r->active == r->path.get()) r->path->Rebuild();
        else {
            if (r->built && r->active) { VHR_CHECK(vhr_context_synchronize(r->resource_manager->ctx)); r->active->DeregisterPath(*r->render_graph, *r->resource_manager); }
            r->path->Build();
        }
        r->active = r->path.get();
        r->built = true;
    });
}

// Switching the active render path to the fully ray-traced one (Renderer's render-path combo box, user_interface.cpp) and its
// "Alpha test for shadows" radio buttons (raytraced_render_path.cpp:80-91) + Rebuild().
int vhrh_set_raytraced_path(vhrh_renderer *r, int use_anyhit_shader) {
    if (!r) return VHR_ERR_INVALID;
    return guarded(r, [&] {
        r->raytraced_path->use_anyhit_shader = use_anyhit_shader != 0;
        if (r->built && r->active == r->raytraced_path.get()) r->raytraced_path->Rebuild();
        else {
            if (r->built && r->active) { VHR_CHECK(vhr_context_synchronize(r->resource_manager->ctx)); r->active->DeregisterPath(*r->render_graph, *r->resource_manager); }
            r->raytraced_path->Build();
        }
        r->active = r->raytraced_path.get();
        r->built = true;
    });
}

// gbuffer_mode 0: the harness has uploaded the G-buffer images itself; 1: run the CUDA primary-ray producer
int vhrh_set_gbuffer_producer(vhrh_renderer *r, int gbuffer_mode) {
    if (!r) return VHR_ERR_INVALID;
    return guarded(r, [&] {
        ResourceManager *rm = r->resource_manager.get();
        if (gbuffer_mode == 1)
            r->render_graph->SetGraphicsPassHook("G-Buffer Pass", [rm](vhr_context *ctx) { VHR_CHECK(vhr_gbuffer_pass(ctx, rm->width, rm->height)); });
        else
            r->render_graph->SetGraphicsPassHook("G-Buffer Pass", [](vhr_context *) {});
    });
}

// shadow_map_mode 0 (the default): no producer, the pass records its draw calls and the harness may upload the Shadow Map itself;
// 1: the CUDA depth rasteriser. The graph binds the pass's attachment ("Shadow Map", binding 0) before the hook runs.
int vhrh_set_shadow_map_producer(vhrh_renderer *r, int shadow_map_mode) {
    if (!r) return VHR_ERR_INVALID;
    return guarded(r, [&] {
        if (shadow_map_mode == 1)
            r->render_graph->SetGraphicsPassHook("Shadow Map Pass", [](vhr_context *ctx) { VHR_CHECK(vhr_shadow_map_pass(ctx)); });
        else
            r->render_graph->SetGraphicsPassHook("Shadow Map Pass", nullptr);
    });
}

// Renderer::Render (renderer.cpp:184-235): UBO update + RenderGraph::Execute; gather = GatherPerformanceStatistics
int vhrh_render(vhrh_renderer *r, const void *per_frame_data, size_t size, int gather_statistics) {
    if (!r || !per_frame_data || size != sizeof(PerFrameData)) return VHR_ERR_INVALID;
    return guarded(r, [&] {
        VHR_ASSERT(r->built, "vhrh_set_modes must be called before rendering");
        PerFrameData pfd;
        memcpy(&pfd, per_frame_data, sizeof(pfd));
        r->resource_manager->UpdatePerFrameUBO(0, pfd);
        r->render_graph->Execute(0);
        if (gather_statistics) r->render_graph->GatherPerformanceStatistics();
    });
}

uint32_t vhrh_execution_order(vhrh_renderer *r, char *buffer, size_t capacity) {
    // passes joined by '\n'; returns the number of passes
    if (!r) return 0;
    std::string s;
    for (const std::string &p : r->render_graph->execution_order) { if (!s.empty()) s += '\n'; s += p; }
    if (buffer && capacity) { strncpy(buffer, s.c_str(), capacity - 1); buffer[capacity - 1] = 0; }
    return (uint32_t)r->render_graph->execution_order.size();
}

// last = 1: last frame's time, 0: the 0.95/0.05 moving average (render_graph.cpp:199); < 0 if unknown
double vhrh_pass_time_ms(vhrh_renderer *r, const char *pass_name, int last) {
    if (!r || !pass_name) return -1.0;
    auto &m = last ? r->render_graph->last_pass_ms : r->render_graph->pass_timestamps;
    auto it = m.find(pass_name);
    return it == m.end() ? -1.0 : it->second;
}

int vhrh_svgf_push_constants(vhrh_renderer *r, void *out24) {
    if (!r || !out24) return VHR_ERR_INVALID;
    memcpy(out24, &r->path->svgf_push_constants, sizeof(SVGFPushConstants));
    return VHR_OK;
}

}  // extern "C"
