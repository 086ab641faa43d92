// vhr_internal.h — host-side context of the C-ABI (not installed; include/vhr_b200.h is the public surface).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/vhr_b200.h"
#include "vhr_common.cuh"

namespace vhr {

struct Image {
    void *ptr = nullptr;
    void *twin = nullptr;      // second buffer of a double-buffered storage image (moments history, SURVEY Q11)
    uint32_t width = 0, height = 0;
    int format = 0;
    size_t bytes = 0;
    bool used = false;
    // transfer-queue state (vhr_image_upload_async / vhr_image_download_async)
    cudaEvent_t upload_done = nullptr;   // recorded on the upload stream after the last asynchronous upload
    bool upload_pending = false;         // the compute stream has not yet waited on upload_done
    void *staging = nullptr;             // device-side snapshot the download stream reads (the image itself may be rewritten)
    cudaEvent_t staged = nullptr;        // snapshot written (compute stream)
    cudaEvent_t staging_free = nullptr;  // snapshot read back (download stream)
    bool staging_busy = false;
    cudaEvent_t direct_read_done = nullptr;   // last vhr_image_download_rows_async (reads the image itself): writers wait for it
    bool direct_read_pending = false;
    // multi-GPU: the same image in the other ranks' HBM, mapped through CUDA IPC (NVLink peer memory); index = rank
    void *peer[VHR_MAX_RANKS] = {};
    void *peer_twin[VHR_MAX_RANKS] = {};
    // copy-free blits (VHR_OPT_BLIT_ALIAS): after blit(src -> dst) both images show ONE buffer (ptr == shares_with->ptr) and the
    // allocation dst gave up waits in `spare` (held by exactly one of the two); whoever is written first takes the spare
    // (make_writable) — the copy a blit would do never happens, the image contents are what a copy would have left.
    Image *shares_with = nullptr;
    void *spare = nullptr;
};

inline int format_texel_bytes(int fmt) {
    switch (fmt) {
        case VHR_FORMAT_B8G8R8A8_UNORM: return 4;
        case VHR_FORMAT_B8G8R8A8_SRGB: return 4;
        case VHR_FORMAT_R16G16_SFLOAT: return 4;
        case VHR_FORMAT_R16G16B16A16_SFLOAT: return 8;
        case VHR_FORMAT_D32_SFLOAT: return 4;
    }
    return 0;
}

// Device-side acceleration structure (bvh_build.cu / trace_kernels.cu)
struct Bvh {
    uint32_t n_tris = 0;
    uint32_t n_nodes2 = 0;         // binary nodes
    uint32_t n_wide = 0;           // 8-wide nodes
    void *wide_nodes = nullptr;    // WideNode[n_wide]
    float4 *tri_verts = nullptr;   // 3 float4 per triangle, leaf order (w of v0 = geometry index bits, w of v1 = primitive id bits)
    void *scratch = nullptr;       // everything else allocated by the build (freed with the Bvh)
    vhr_bvh_stats stats = {};
};

struct Options {
    int ao_spp = 2;
    int trace_shadows = 1;
    int trace_ao = 1;
    int trace_reflections = 1;
    int row_begin = 0;
    int row_end = -1;            // -1 = image height
    int svgf_fused = 0;
    int blit_alias = 0;          // 1: same-size blits alias buffers copy-on-write instead of copying (VHR_OPT_BLIT_ALIAS)
    int atrous_variant = 2;      // 0 = direct-load reference-like kernel, 1 = shared-memory tiled kernel, 2 = pixel-pair packed kernel
    int debug_refl_t = 0;        // 1: the ray pass also writes the reflection ray's hit distance (tests)
    int raytraced_alpha_test = 0; // the fully ray-traced path's use_anyhit_shader (raytraced_render_path.h:14)
    int raygen_variant = 0;      // 0 (default, fastest as measured): one thread per pixel, ray kinds in lock step; 1-4: see VHR_OPT_RAYGEN_VARIANT
    int output_rank = -1;        // the rank whose render output the composition passes gather the partitioned frame into; -1 = off (VHR_OPT_OUTPUT_RANK)
};

// Row partition of one frame over the GPUs of a box (vhr_set_partition)
struct Partition {
    bool enabled = false;
    int world = 1, rank = 0;
    int band_begin[VHR_MAX_RANKS + 1] = {};
    int ray_block_rows = 0;
    int motion_halo = 8;
    int no_exchange_step = 16;
};
// What a kernel needs to push its boundary rows into the neighbours' copies of the image it writes
// Scratch of the shadow-map pass (shadow_map_kernels.cu): grows to the largest scene seen, freed with the context
struct ShadowScratch {
    void *counts = nullptr, *offsets = nullptr;      // uint64 per triangle + 1: tile counts and their exclusive scan
    void *clip_list = nullptr;                       // uint32: [0] count, then the triangles that reach beyond the guard band
    void *records = nullptr;                         // 48 B per triangle (written for large triangles only)
    void *scan_tmp = nullptr;                        // CUB scan temporary storage
    size_t counts_bytes = 0, offsets_bytes = 0, clip_list_bytes = 0, records_bytes = 0, scan_tmp_bytes = 0;
    int sms = 0;
    std::vector<void *> retired;                     // buffers a partitioned pass outgrew: freed without a device synchronisation later
};
struct HaloPush {
    void *up = nullptr;       // same image on rank-1 (nullptr: no neighbour / no push)
    void *down = nullptr;     // same image on rank+1
    int rows = 0;             // output rows [y_begin, y_begin+rows) go up, [y_end-rows, y_end) go down
};

}  // namespace vhr

struct vhr_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    uint32_t width = 0, height = 0;
    std::unordered_map<std::string, vhr::Image> transient;
    std::vector<vhr::Image> storage;               // VHR_MAX_GLOBAL_RESOURCES slots
    vhr::Image *bound[VHR_MAX_PASS_BINDINGS] = {};
    uint32_t n_bound = 0;
    vhr::PerFrameData pfd = {};
    bool pfd_set = false;
    // geometry (global vertex / index / primitive buffers, resource_manager.cpp:13-28)
    vhr::Vertex *d_vertices = nullptr;
    uint32_t *d_indices = nullptr;
    vhr::Primitive *d_primitives = nullptr;
    uint32_t n_vertices = 0, n_indices = 0, n_primitives = 0;
    float *d_normal_mats = nullptr;                // 9 floats per primitive: inverseTranspose(mat3(transform)), column-major
    // textures[] (descriptor set 0 binding 4): device table of VHR_MAX_GLOBAL_RESOURCES descriptors + the texel buffers behind it
    vhr::TextureDesc *d_textures = nullptr;
    std::vector<vhr::TextureDesc> textures;        // host mirror; texels == nullptr marks a free slot (resource_manager.cpp:821-824)
    float *d_texel_lut = nullptr;                  // 512 floats: UNORM8 -> float, sRGB8 -> linear float
    float *d_refl_t = nullptr;                     // optional debug image: reflection-ray hit distance per pixel
    uint32_t *d_ray_queue = nullptr;               // head of the persistent ray kernel's pixel queue
    // ssao.comp / ssr.comp: the 2x2 bilinear footprint of every depth texel, one 16-byte word (ssao_kernels.cu); one buffer per queue, so
    // that a screen-space pass recorded on queue 1 does not rebuild the image a pass on queue 0 is still gathering from
    float4 *d_depth_quads[2] = {nullptr, nullptr};
    size_t depth_quads_texels[2] = {0, 0};
    // ssr.comp: (min, max) depth over every 8 x 8-texel tile + a 2-texel apron (ssr_kernels.cu: conservative skip of march steps)
    float2 *d_depth_tiles[2] = {nullptr, nullptr};
    size_t depth_tiles_count[2] = {0, 0};
    int raygen_blocks = 0;                         // resident grid of the persistent ray kernel (SMs x blocks/SM)
    vhr::Bvh bvh;
    vhr::ShadowScratch shadow;
    vhr::Options opt;
    uint64_t launches = 0;
    uint32_t debug_label_depth = 0;                // open vhr_cmd_begin_debug_label ranges
    // VHR_OPT_SVGF_FUSED: svgf.comp's dispatch has already produced a-trous iteration 0 for these storage slots; the step-1
    // dispatch that follows it in the reference's sequence finds this note and launches nothing. `epoch` counts the calls that can
    // change an image, a binding or the per-frame constants: the note only holds for the very next such call.
    uint64_t epoch = 0;
    struct { bool valid = false; int in_slot = -1, out_slot = -1; uint64_t epoch = 0; } fused_it0;
    std::vector<cudaEvent_t> queries;              // timestamp query pool
    // transfer queues: copies that overlap the compute stream (the reference's frames in flight, renderer.cpp:103-108)
    cudaStream_t upload_stream = nullptr, download_stream = nullptr;
    cudaEvent_t compute_tail = nullptr;            // scratch event: "everything enqueued on the compute stream so far"
    std::vector<cudaEvent_t> tickets;              // ring of download-completion events
    uint32_t next_ticket = 0;
    // two queues (vhr_select_queue): `stream` is the selected one
    cudaStream_t queue[2] = {nullptr, nullptr};    // [0] the stream given at creation (or the context's own), [1] created on first use
    cudaEvent_t semaphores[VHR_MAX_SEMAPHORES] = {};
    bool semaphore_signalled[VHR_MAX_SEMAPHORES] = {};
    // multi-GPU partition + peer synchronisation (peer.cu)
    vhr::Partition part;
    uint32_t *sync_flags = nullptr;                       // device: [0, MAX) ray-pass arrivals, [MAX, 2 MAX) halo arrivals, by source rank
    uint32_t *peer_flags[VHR_MAX_RANKS] = {};             // the other ranks' sync_flags (IPC mapped)
    uint32_t seq_ray = 0, seq_halo = 0;
    vhr::Image *gbuffer_peer_written[4] = {};             // the images the last partitioned G-buffer pass stored to every rank (none: cleared by vhr_set_partition)
    std::vector<void *> ipc_opened;                       // everything cudaIpcOpenMemHandle returned (closed with the context)
};

namespace vhr {

// error plumbing (vhr_api.cu)
int fail(int status, const char *fmt, ...);
#define VHR_CUDA_CHECK(expr)                                                                            \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) return vhr::fail(VHR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,           \
                                                 cudaGetErrorString(e__), __FILE__, __LINE__);           \
    } while (0)

// kernel launchers (svgf_kernels.cu, ssao_kernels.cu, trace_kernels.cu, bvh_build.cu); all return a vhr_status
int launch_svgf_temporal(vhr_context *ctx, uint32_t xg, uint32_t yg, const SVGFPushConstants &pc);
int launch_svgf_atrous(vhr_context *ctx, uint32_t xg, uint32_t yg, const SVGFPushConstants &pc);
int launch_ssao(vhr_context *ctx, uint32_t xg, uint32_t yg, float radius);
int build_depth_quads(vhr_context *ctx, const float *depth, int W, int H, const float4 **quads);     // -> the selected queue's quad image (ssao_kernels.cu)
int launch_ssao_blur(vhr_context *ctx, uint32_t xg, uint32_t yg);
int launch_ssr(vhr_context *ctx, uint32_t xg, uint32_t yg, const SSRPushConstants &pc);
int launch_trace_rays(vhr_context *ctx, uint32_t width, uint32_t height);
int launch_gbuffer(vhr_context *ctx, uint32_t width, uint32_t height);
int launch_raytraced(vhr_context *ctx, uint32_t width, uint32_t height);
int launch_present(vhr_context *ctx);
int launch_composition(vhr_context *ctx, int shadow_mode, int ao_mode, int reflection_mode);
int launch_shadow_map(vhr_context *ctx);        // shadow_map_kernels.cu
void free_shadow_scratch(vhr_context *ctx);
int launch_trace_explicit(vhr_context *ctx, const float *rays, uint32_t n, int any_hit, float *out_t, uint32_t *out_ids,
                          float *out_uv);
int launch_shade_hits(vhr_context *ctx, int kind, const vhr_shade_record *records, uint32_t n, uint32_t *out);   // records validated
// peer.cu: stream-ordered flag exchange with the other ranks (cuStreamWriteValue32 / cuStreamWaitValue32)
int peer_sync_neighbours(vhr_context *ctx);   // after a kernel that pushed halo rows: tell both neighbours, wait for theirs
int peer_sync_all(vhr_context *ctx);          // after the ray pass scattered its rows to their owners: all ranks <-> all ranks
HaloPush halo_push_for(vhr_context *ctx, Image *out, bool twin, int rows);
void peer_close_all(vhr_context *ctx);
// Call before enqueueing work that writes `im`: an image that shares its buffer with a blit partner gets the spare allocation
// (its old content is copied over first unless the write covers the `whole` image). No-op for images that share nothing.
int make_writable(vhr_context *ctx, Image *im, bool whole);
// "'name'" of a transient image, "storage image <slot>" of a storage image (error messages)
std::string image_label(vhr_context *ctx, const Image *im);
// does a pass dispatched over xg x yg groups of 8 x 8 (or a w x h launch) overwrite every texel of `im`?
inline bool covers_image(const vhr_context *ctx, const Image *im, uint64_t w, uint64_t h) {
    return !ctx->part.enabled && ctx->opt.row_begin <= 0 && (ctx->opt.row_end < 0 || ctx->opt.row_end >= (int)im->height) && w >= im->width && h >= im->height;
}
int build_bvh(vhr_context *ctx);
void free_bvh(vhr_context *ctx);

inline Image *storage_slot(vhr_context *ctx, int slot) {
    if (slot < 0 || slot >= VHR_MAX_GLOBAL_RESOURCES) return nullptr;
    Image &im = ctx->storage[slot];
    return im.used ? &im : nullptr;
}

}  // namespace vhr
