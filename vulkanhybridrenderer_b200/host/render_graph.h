// render_graph.h — B200 host mirror of the reference's render-graph boundary (the seam HybridRenderPath talks to).
//
//   ResourceManager            <- src/rendering_backend/resource_manager.{h,cpp}  (UpdateGeometry :291, UpdatePerFrameUBO :362,
//                                 UploadNewStorageImage :230, DestroyStorageImage :265) — now a thin owner of a vhr_context
//   RenderGraph                <- src/render_graph/render_graph.{h,cpp} (Add*Pass :70-116, Build :118, FindExecutionOrder :686,
//                                 Execute :151, GatherPerformanceStatistics :189, DestroyResources :16)
//   ComputeExecutionContext    <- src/render_graph/compute_execution_context.{h,cpp}
//   RaytracingExecutionContext <- src/render_graph/raytracing_execution_context.{h,cpp}
//   GraphicsExecutionContext   <- src/render_graph/graphics_execution_context.{h,cpp}: rasterisation is outside the hot
//                                 path; graphics passes stay in the graph as external producers / consumers (a hook runs
//                                 whatever fills or reads their images, e.g. the CUDA primary-ray G-buffer pass).
// Scheduling is the reference's (BFS back from the writer of RENDER_OUTPUT); barriers are CUDA stream order; per-pass
// timestamps are CUDA events with the reference's 0.95/0.05 moving average.
#pragma once
#include <unordered_map>

#include "host_types.h"

class ResourceManager {
public:
    // One context = one GPU + one stream (VulkanContext + ResourceManager constructors, renderer.cpp:18-21).
    ResourceManager(int device, void *cuda_stream, uint32_t width, uint32_t height);
    ~ResourceManager();
    ResourceManager(const ResourceManager &) = delete;

    void UpdateGeometry(std::vector<Vertex> &vertices, std::vector<uint32_t> &indices, Scene &scene);
    void UpdatePerFrameUBO(uint32_t resource_idx, PerFrameData &per_frame_data);
    // resource_manager.cpp:152-193 (+ GetSampler :880-910): tightly packed R8G8B8A8 texels -> slot of textures[]
    uint32_t UploadTextureFromData(uint32_t width, uint32_t height, uint8_t *data, VkFormat format = VK_FORMAT_R8G8B8A8_UNORM,
                                   SamplerInfo *sampler_info = nullptr);
    uint32_t UploadNewStorageImage(uint32_t width, uint32_t height, VkFormat format);
    void DestroyStorageImage(uint32_t image_idx);

    vhr_context *ctx = nullptr;
    Scene scene;
    uint32_t width, height;
};

class RenderGraph;

class ComputeExecutionContext {
public:
    ComputeExecutionContext(RenderGraph &render_graph, ResourceManager &resource_manager, const RenderPassDescription &pass)
        : render_graph(render_graph), resource_manager(resource_manager), pass(pass) {}
    glmlite::uvec2 GetDisplaySize();
    void Dispatch(const char *shader, uint32_t x_groups, uint32_t y_groups, uint32_t z_groups);
    template <typename T>
    void Dispatch(const char *shader, uint32_t x_groups, uint32_t y_groups, uint32_t z_groups, T &push_constants) {
        DispatchRaw(shader, x_groups, y_groups, z_groups, &push_constants, sizeof(T));
    }
    void BlitImageStorageToTransient(int src, const char *dst);
    void BlitImageTransientToStorage(const char *src, int dst);
    void BlitImageStorageToStorage(int src, int dst);

private:
    void DispatchRaw(const char *shader, uint32_t x_groups, uint32_t y_groups, uint32_t z_groups, const void *pc, size_t pc_size);
    RenderGraph &render_graph;
    ResourceManager &resource_manager;
    const RenderPassDescription &pass;
};

class RaytracingExecutionContext {
public:
    RaytracingExecutionContext(ResourceManager &resource_manager, const char *pipeline) : resource_manager(resource_manager), pipeline(pipeline) {}
    void TraceRays(uint32_t width, uint32_t height);

private:
    ResourceManager &resource_manager;
    const char *pipeline;
};

class GraphicsExecutionContext {
public:
    // `pipeline` is the graphics pipeline being executed (graphics_execution_context.h:6-10); nullptr for the counting
    // context used when a rasterised pass has no CUDA counterpart.
    explicit GraphicsExecutionContext(ResourceManager &resource_manager, const GraphicsPipelineDescription *pipeline = nullptr)
        : resource_manager(resource_manager), pipeline(pipeline) {}
    // Geometry draw calls have no CUDA counterpart; they are accepted and counted so RegisterPath runs unchanged.
    void BindGlobalVertexAndIndexBuffers() {}
    template <typename T> void PushConstants(T &) {}
    void DrawIndexed(uint32_t, uint32_t, uint32_t, uint32_t, uint32_t) { ++draws; }
    // graphics_execution_context.cpp:38-41. For a pipeline whose fragment shader has a CUDA kernel (the composition
    // pass) this launches it through vhr_draw; otherwise the call only counts.
    void Draw(uint32_t vertex_count, uint32_t instance_count, uint32_t first_vertex, uint32_t first_instance);
    static bool HasKernel(const GraphicsPipelineDescription &pipeline);
    uint32_t draws = 0;
    ResourceManager &resource_manager;
    const GraphicsPipelineDescription *pipeline;
};

class RenderGraph {
public:
    explicit RenderGraph(ResourceManager &resource_manager);
    void DestroyResources();

    void AddGraphicsPass(const char *render_pass_name, std::vector<TransientResource> dependencies, std::vector<TransientResource> outputs,
                         std::vector<GraphicsPipelineDescription> pipelines, GraphicsPassCallback callback);
    void AddRaytracingPass(const char *render_pass_name, std::vector<TransientResource> dependencies, std::vector<TransientResource> outputs,
                           RaytracingPipelineDescription pipeline, RaytracingPassCallback callback);
    void AddComputePass(const char *render_pass_name, std::vector<TransientResource> dependencies, std::vector<TransientResource> outputs,
                        ComputePipelineDescription pipeline, ComputePassCallback callback);

    void Build();
    void Execute(uint32_t resource_idx);
    void GatherPerformanceStatistics();
    bool ContainsImage(const std::string &image_name) const;
    VkFormat GetImageFormat(const std::string &image_name) const;

    // What replaces the rasteriser for a graphics pass: called instead of recording draw calls (e.g. the CUDA G-buffer
    // producer for "G-Buffer Pass"; nothing for "Composition Pass" when only the hot path is exercised). An empty `hook` removes
    // the pass's hook: its draw calls are recorded again.
    void SetGraphicsPassHook(const std::string &pass_name, std::function<void(vhr_context *)> hook);

    std::vector<std::string> execution_order;
    std::unordered_map<std::string, double> pass_timestamps;      // EMA, ms (render_graph.cpp:199)
    std::unordered_map<std::string, double> last_pass_ms;         // last frame, ms

private:
    friend class ComputeExecutionContext;
    void ActualizeResource(const TransientResource &resource, const char *render_pass_name);
    void FindExecutionOrder();
    bool SanityCheck();
    void BindPassImages(const RenderPassDescription &pass);

    ResourceManager &resource_manager;
    std::vector<std::string> declaration_order;
    std::unordered_map<std::string, std::vector<std::string>> readers, writers;
    std::unordered_map<std::string, RenderPassDescription> pass_descriptions;
    std::unordered_map<std::string, TransientImage> images;
    std::unordered_map<std::string, std::string> compute_kernels;   // shader path -> owning pass (render_graph.cpp:676-681)
    std::unordered_map<std::string, std::function<void(vhr_context *)>> graphics_hooks;
    bool timestamps_pending = false;
};
