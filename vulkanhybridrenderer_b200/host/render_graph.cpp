// render_graph.cpp — see render_graph.h. Written against the behaviour of the reference files cited there; the
// implementation is CUDA-stream based (no command buffers, descriptor sets, layouts or barriers exist here).
#include "render_graph.h"

#include <algorithm>
#include <deque>

// ---- ResourceManager ---------------------------------------------------------------------------------------------
ResourceManager::ResourceManager(int device, void *cuda_stream, uint32_t w, uint32_t h) : width(w), height(h) {
    VHR_CHECK(vhr_context_create(device, cuda_stream, w, h, &ctx));
}
ResourceManager::~ResourceManager() { vhr_context_destroy(ctx); }

void ResourceManager::UpdateGeometry(std::vector<Vertex> &vertices, std::vector<uint32_t> &indices, Scene &new_scene) {
    // resource_manager.cpp:607-644: one geometry per primitive, flattened in mesh order; that flat index is the
    // G-buffer object id and gl_GeometryIndexEXT.
    std::vector<Primitive> flat;
    for (Mesh &mesh : new_scene.meshes)
        for (Primitive &p : mesh.primitives) flat.push_back(p);
    VHR_CHECK(vhr_update_geometry(ctx, vertices.data(), (uint32_t)vertices.size(), indices.data(), (uint32_t)indices.size(), flat.data(),
                                  (uint32_t)flat.size()));
    scene = new_scene;
}
void ResourceManager::UpdatePerFrameUBO(uint32_t, PerFrameData &per_frame_data) {
    VHR_CHECK(vhr_update_per_frame_ubo(ctx, &per_frame_data, sizeof(PerFrameData)));
}
uint32_t ResourceManager::UploadTextureFromData(uint32_t w, uint32_t h, uint8_t *data, VkFormat format, SamplerInfo *sampler_info) {
    vhr_sampler_info si{};
    if (sampler_info) si = vhr_sampler_info{sampler_info->mag_filter, sampler_info->min_filter, sampler_info->address_mode_u, sampler_info->address_mode_v};
    int slot = vhr_upload_texture_from_data(ctx, w, h, data, (int)format, sampler_info ? &si : nullptr);
    if (slot < 0) throw VhrHostError{slot, std::string("UploadTextureFromData: ") + vhr_last_error()};
    return (uint32_t)slot;
}
uint32_t ResourceManager::UploadNewStorageImage(uint32_t w, uint32_t h, VkFormat format) {
    int slot = vhr_upload_new_storage_image(ctx, w, h, (int)format);
    if (slot < 0) throw VhrHostError{slot, std::string("UploadNewStorageImage: ") + vhr_last_error()};
    return (uint32_t)slot;
}
void ResourceManager::DestroyStorageImage(uint32_t image_idx) { VHR_CHECK(vhr_destroy_storage_image(ctx, (int)image_idx)); }

// ---- execution contexts --------------------------------------------------------------------------------------------
glmlite::uvec2 ComputeExecutionContext::GetDisplaySize() {
    glmlite::uvec2 s{0, 0};
    VHR_CHECK(vhr_get_display_size(resource_manager.ctx, &s.x, &s.y));
    return s;
}
void ComputeExecutionContext::DispatchRaw(const char *shader, uint32_t xg, uint32_t yg, uint32_t zg, const void *pc, size_t pc_size) {
    // compute_execution_context.cpp:13: the kernel must have been registered by the pass being executed
    auto it = render_graph.compute_kernels.find(shader);
    VHR_ASSERT(it != render_graph.compute_kernels.end() && it->second == pass.name, std::string("kernel not registered by this pass: ") + shader);
    const ComputePassDescription &d = std::get<ComputePassDescription>(pass.description);
    // compute_execution_context.h:23: assert(sizeof(T) == pipeline.push_constant_description.size)
    VHR_ASSERT(pc == nullptr || pc_size == d.pipeline_description.push_constant_description.size, "push constant size differs from the declared size");
    VHR_CHECK(vhr_dispatch(resource_manager.ctx, shader, xg, yg, zg, pc, pc_size));
}
void ComputeExecutionContext::Dispatch(const char *shader, uint32_t xg, uint32_t yg, uint32_t zg) { DispatchRaw(shader, xg, yg, zg, nullptr, 0); }
void ComputeExecutionContext::BlitImageStorageToTransient(int src, const char *dst) { VHR_CHECK(vhr_blit_storage_to_transient(resource_manager.ctx, src, dst)); }
void ComputeExecutionContext::BlitImageTransientToStorage(const char *src, int dst) { VHR_CHECK(vhr_blit_transient_to_storage(resource_manager.ctx, src, dst)); }
void ComputeExecutionContext::BlitImageStorageToStorage(int src, int dst) { VHR_CHECK(vhr_blit_storage_to_storage(resource_manager.ctx, src, dst)); }

void RaytracingExecutionContext::TraceRays(uint32_t w, uint32_t h) { VHR_CHECK(vhr_trace_rays(resource_manager.ctx, pipeline, w, h)); }

// ---- RenderGraph ---------------------------------------------------------------------------------------------------
RenderGraph::RenderGraph(ResourceManager &rm) : resource_manager(rm) {}

void RenderGraph::DestroyResources() {
    VHR_CHECK(vhr_destroy_transient_resources(resource_manager.ctx));
    execution_order.clear(); declaration_order.clear();
    readers.clear(); writers.clear(); pass_descriptions.clear(); images.clear(); compute_kernels.clear();
    pass_timestamps.clear(); last_pass_ms.clear();
    timestamps_pending = false;
}

void RenderGraph::AddGraphicsPass(const char *name, std::vector<TransientResource> deps, std::vector<TransientResource> outs,
                                  std::vector<GraphicsPipelineDescription> pipelines, GraphicsPassCallback callback) {
    VHR_ASSERT(!pass_descriptions.count(name), std::string("duplicate pass name: ") + name);   // render_graph.cpp:83
    pass_descriptions[name] = RenderPassDescription{name, std::move(deps), std::move(outs), GraphicsPassDescription{std::move(pipelines), std::move(callback)}};
    declaration_order.push_back(name);
}
void RenderGraph::AddRaytracingPass(const char *name, std::vector<TransientResource> deps, std::vector<TransientResource> outs,
                                    RaytracingPipelineDescription pipeline, RaytracingPassCallback callback) {
    VHR_ASSERT(!pass_descriptions.count(name), std::string("duplicate pass name: ") + name);   // render_graph.cpp:99
    pass_descriptions[name] = RenderPassDescription{name, std::move(deps), std::move(outs), RaytracingPassDescription{std::move(pipeline), std::move(callback)}};
    declaration_order.push_back(name);
}
void RenderGraph::AddComputePass(const char *name, std::vector<TransientResource> deps, std::vector<TransientResource> outs,
                                 ComputePipelineDescription pipeline, ComputePassCallback callback) {
    VHR_ASSERT(!pass_descriptions.count(name), std::string("duplicate pass name: ") + name);   // render_graph.cpp:114
    pass_descriptions[name] = RenderPassDescription{name, std::move(deps), std::move(outs), ComputePassDescription{std::move(pipeline), std::move(callback)}};
    declaration_order.push_back(name);
}

void RenderGraph::ActualizeResource(const TransientResource &resource, const char *pass_name) {
    VHR_ASSERT(resource.type == TransientResourceType::Image, "only image resources are supported");   // render_graph.cpp:922
    const TransientImage &img = resource.image;
    auto it = images.find(resource.name);
    if (it == images.end()) {
        images[resource.name] = img;
    } else {
        // RenderGraph::SanityCheck (render_graph.cpp:980-1021): one name, one extent, one format
        VHR_ASSERT(it->second.width == img.width && it->second.height == img.height && it->second.format == img.format,
                   std::string("image '") + resource.name + "' re-declared with another size/format by pass " + pass_name);
    }
    VHR_CHECK(vhr_actualize_image(resource_manager.ctx, resource.name, img.width, img.height, (int)img.format));
}

void RenderGraph::Build() {
    readers.clear(); writers.clear(); compute_kernels.clear();
    for (const std::string &name : declaration_order) {
        RenderPassDescription &pass = pass_descriptions[name];
        for (TransientResource &r : pass.dependencies) { readers[r.name].push_back(name); ActualizeResource(r, pass.name); }
        for (TransientResource &r : pass.outputs) { writers[r.name].push_back(name); ActualizeResource(r, pass.name); }
        if (auto *c = std::get_if<ComputePassDescription>(&pass.description)) {
            for (const ComputeKernel &k : c->pipeline_description.kernels) {
                VHR_ASSERT(!compute_kernels.count(k.shader), std::string("compute kernel registered twice: ") + k.shader);   // render_graph.cpp:677
                compute_kernels[k.shader] = name;
            }
        }
    }
    FindExecutionOrder();
    VHR_ASSERT(SanityCheck(), "render graph sanity check failed");
    VHR_CHECK(vhr_create_query_pool(resource_manager.ctx, (uint32_t)execution_order.size() * 2));   // render_graph.cpp:143-148
    timestamps_pending = false;
}

void RenderGraph::FindExecutionOrder() {
    // render_graph.cpp:686-720: breadth-first from the single writer of RENDER_OUTPUT back through the writers of every
    // dependency; reverse; keep the first occurrence of each pass.
    VHR_ASSERT(writers["RENDER_OUTPUT"].size() == 1, "exactly one pass must write RENDER_OUTPUT");
    std::vector<std::string> order{writers["RENDER_OUTPUT"][0]};
    std::deque<std::string> frontier{order[0]};
    size_t guard = 0;
    while (!frontier.empty()) {
        const RenderPassDescription &pass = pass_descriptions[frontier.front()];
        frontier.pop_front();
        for (const TransientResource &dep : pass.dependencies)
            for (const std::string &w : writers[dep.name]) {
                order.push_back(w);
                frontier.push_back(w);
            }
        VHR_ASSERT(++guard < 100000, "cycle in the render graph");
    }
    std::reverse(order.begin(), order.end());
    execution_order.clear();
    for (const std::string &p : order)
        if (std::find(execution_order.begin(), execution_order.end(), p) == execution_order.end()) execution_order.push_back(p);
}

bool RenderGraph::SanityCheck() {
    // every dependency has a writer or is fed from outside by a graphics hook; bindings inside a pass are unique
    for (const std::string &name : execution_order) {
        const RenderPassDescription &pass = pass_descriptions[name];
        std::vector<uint32_t> seen;
        auto check = [&](const std::vector<TransientResource> &v) {
            for (const TransientResource &r : v) {
                if (std::find(seen.begin(), seen.end(), r.image.binding) != seen.end()) return false;
                seen.push_back(r.image.binding);
            }
            return true;
        };
        // graphics passes number their attachments from 0 independently of the sampled inputs (vulkan_utils.h:347-453)
        if (std::holds_alternative<GraphicsPassDescription>(pass.description)) {
            if (!check(pass.dependencies)) return false;
            seen.clear();
            if (!check(pass.outputs)) return false;
        } else if (!check(pass.dependencies) || !check(pass.outputs)) {
            return false;
        }
    }
    return true;
}

void RenderGraph::BindPassImages(const RenderPassDescription &pass) {
    // descriptor set 3 = dependencies then outputs, addressed by `binding` (render_graph.cpp:603-664)
    const char *names[VHR_MAX_PASS_BINDINGS] = {};
    uint32_t count = 0;
    auto put = [&](const std::vector<TransientResource> &v) {
        for (const TransientResource &r : v) {
            VHR_ASSERT(r.image.binding < VHR_MAX_PASS_BINDINGS, "binding index too large");
            names[r.image.binding] = r.name;
            count = std::max(count, r.image.binding + 1);
        }
    };
    put(pass.dependencies);
    put(pass.outputs);
    for (uint32_t i = 0; i < count; ++i) VHR_ASSERT(names[i] != nullptr, std::string("pass '") + pass.name + "' leaves a binding gap");
    VHR_CHECK(vhr_bind_pass_images(resource_manager.ctx, names, count));
}

bool GraphicsExecutionContext::HasKernel(const GraphicsPipelineDescription &pipeline) {
    if (!pipeline.fragment_shader) return false;
    const std::string fs = pipeline.fragment_shader;
    return fs == "hybrid_render_path/composition.frag" || fs == "raytraced_render_path/composition.frag";
}
void GraphicsExecutionContext::Draw(uint32_t vertex_count, uint32_t instance_count, uint32_t first_vertex, uint32_t first_instance) {
    ++draws;
    if (!pipeline || !HasKernel(*pipeline)) return;
    const std::vector<int> &sc = pipeline->specialization_constants;
    std::vector<int32_t> constants(sc.begin(), sc.end());
    VHR_CHECK(vhr_draw(resource_manager.ctx, pipeline->fragment_shader, constants.data(), (uint32_t)constants.size(), vertex_count, instance_count,
                       first_vertex, first_instance));
}

void RenderGraph::SetGraphicsPassHook(const std::string &pass_name, std::function<void(vhr_context *)> hook) {
    if (hook) graphics_hooks[pass_name] = std::move(hook);
    else graphics_hooks.erase(pass_name);
}

void RenderGraph::Execute(uint32_t resource_idx) {
    (void)resource_idx;   // the reference's 3 frames in flight collapse to stream order
    vhr_context *ctx = resource_manager.ctx;
    for (size_t i = 0; i < execution_order.size(); ++i) {
        const RenderPassDescription &pass = pass_descriptions[execution_order[i]];
        VHR_CHECK(vhr_cmd_begin_debug_label(ctx, pass.name));      // render_graph.cpp:160-164
        VHR_CHECK(vhr_write_timestamp(ctx, (uint32_t)i * 2));
        if (auto *g = std::get_if<GraphicsPassDescription>(&pass.description)) {
            auto hook = graphics_hooks.find(pass.name);
            if (hook != graphics_hooks.end()) {
                // graphics passes bind only their attachments (outputs) for an external producer
                const char *names[VHR_MAX_PASS_BINDINGS] = {};
                uint32_t count = 0;
                for (const TransientResource &r : pass.outputs) { names[r.image.binding] = r.name; count = std::max(count, r.image.binding + 1); }
                VHR_CHECK(vhr_bind_pass_images(ctx, names, count));
                hook->second(ctx);
            } else {
                // Pipelines whose fragment shader exists as a CUDA kernel (the composition pass) execute for real: sampled
                // inputs by binding, colour attachments after them. For the rest there is no rasteriser in this build:
                // the draw-call recording runs against a counting context so the path's lambdas execute exactly as in the
                // reference, and the result is dropped.
                bool bound = false;
                g->callback([&](std::string pipeline_name, GraphicsExecutionCallback cb) {
                    const GraphicsPipelineDescription *pipeline = nullptr;
                    for (const GraphicsPipelineDescription &d : g->pipeline_descriptions)
                        if (pipeline_name == d.name) pipeline = &d;
                    VHR_ASSERT(pipeline != nullptr, "unknown graphics pipeline: " + pipeline_name);      // render_graph.cpp:738
                    if (GraphicsExecutionContext::HasKernel(*pipeline)) {
                        if (!bound) {
                            const char *names[VHR_MAX_PASS_BINDINGS] = {};
                            uint32_t count = 0, n_sampled = 0;
                            for (const TransientResource &r : pass.dependencies) { names[r.image.binding] = r.name; n_sampled = std::max(n_sampled, r.image.binding + 1); }
                            count = n_sampled;
                            for (const TransientResource &r : pass.outputs) {
                                VHR_ASSERT(n_sampled + r.image.binding < VHR_MAX_PASS_BINDINGS, "too many graphics-pass images");
                                names[n_sampled + r.image.binding] = r.name;
                                count = std::max(count, n_sampled + r.image.binding + 1);
                            }
                            for (uint32_t k = 0; k < count; ++k) VHR_ASSERT(names[k] != nullptr, std::string("pass '") + pass.name + "' leaves a binding gap");
                            VHR_CHECK(vhr_bind_pass_images(ctx, names, count));
                            bound = true;
                        }
                        GraphicsExecutionContext ec(resource_manager, pipeline);
                        cb(ec);
                    } else {
                        GraphicsExecutionContext ec(resource_manager);
                        cb(ec);
                    }
                });
            }
        } else if (auto *r = std::get_if<RaytracingPassDescription>(&pass.description)) {
            BindPassImages(pass);
            r->callback([&](std::string pipeline_name, RaytracingExecutionCallback cb) {
                VHR_ASSERT(pipeline_name == r->pipeline_description.name, "unknown ray-tracing pipeline: " + pipeline_name);
                RaytracingExecutionContext ec(resource_manager, r->pipeline_description.name);
                cb(ec);
            });
        } else {
            auto &c = std::get<ComputePassDescription>(pass.description);
            BindPassImages(pass);
            ComputeExecutionContext ec(*this, resource_manager, pass);
            c.callback(ec);
        }
        VHR_CHECK(vhr_write_timestamp(ctx, (uint32_t)i * 2 + 1));
        VHR_CHECK(vhr_cmd_end_debug_label(ctx));                             // render_graph.cpp:184
    }
    timestamps_pending = true;
}

void RenderGraph::GatherPerformanceStatistics() {
    if (!timestamps_pending) return;
    for (size_t i = 0; i < execution_order.size(); ++i) {
        double ms = 0.0;
        VHR_CHECK(vhr_get_query_elapsed_ms(resource_manager.ctx, (uint32_t)i * 2, (uint32_t)i * 2 + 1, &ms));   // blocks, like VK_QUERY_RESULT_WAIT_BIT
        const std::string &name = execution_order[i];
        last_pass_ms[name] = ms;
        pass_timestamps[name] = pass_timestamps[name] * 0.95 + ms * 0.05;   // render_graph.cpp:199
    }
    timestamps_pending = false;
}

bool RenderGraph::ContainsImage(const std::string &n) const { return images.count(n) != 0; }
VkFormat RenderGraph::GetImageFormat(const std::string &n) const {
    auto it = images.find(n);
    return it == images.end() ? VK_FORMAT_UNDEFINED : it->second.format;
}
