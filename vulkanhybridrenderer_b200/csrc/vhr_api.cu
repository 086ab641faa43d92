// vhr_api.cu — the C-ABI of include/vhr_b200.h: context, image tables, per-frame constants, pass dispatch.
// Each entry point cites the reference call it replaces in the header.
#include <stdarg.h>
#include <stdio.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "vhr_internal.h"

// NVTX ranges (header-only nvtx3; visible in Nsight Systems / Compute): one range per pass node (vhr_cmd_begin_debug_label, the
// counterpart of the vkCmdBeginDebugUtilsLabelEXT per pass at render_graph.cpp:160-164) and one per kernel-launching entry point,
// named after the reference's shader path / pipeline name.
#include <nvtx3/nvToolsExt.h>
namespace {
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name ? name : "(null)"); }
    ~NvtxRange() { nvtxRangePop(); }
};
}  // namespace

namespace vhr {

static thread_local char g_error[512] = "";

int fail(int status, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
    return status;
}

static int alloc_image(vhr_context *ctx, Image &im, uint32_t w, uint32_t h, int fmt) {
    int tb = format_texel_bytes(fmt);
    if (!tb) return fail(VHR_ERR_INVALID, "unsupported VkFormat %d", fmt);
    if (w == 0 || h == 0) return fail(VHR_ERR_INVALID, "image size %ux%u", w, h);
    im.width = w; im.height = h; im.format = fmt;
    im.bytes = (size_t)w * h * tb;
    if (ctx->device >= 0) {    // a VHR_DEVICE_NONE context only keeps the image table (graph building / validation)
        // 16 rows of zero padding behind the image: the TMA view (x, row mod S, row div S) of the a-trous kernel reads the
        // whole last slab, i.e. up to S - 1 <= 15 rows past the image, and those must read as "no texel"
        const size_t padded = im.bytes + (size_t)16 * w * tb;
        VHR_CUDA_CHECK(cudaMalloc(&im.ptr, padded));
        VHR_CUDA_CHECK(cudaMemsetAsync(im.ptr, 0, padded, ctx->stream));
    }
    im.twin = nullptr;
    im.used = true;
    return VHR_OK;
}
static void free_image(Image &im) {
    if (im.shares_with) {          // the partner keeps the shared buffer; the idle allocation goes
        Image *o = im.shares_with;
        void *sp = im.spare ? im.spare : o->spare;
        if (sp) cudaFree(sp);
        o->spare = nullptr; o->shares_with = nullptr;
        im.ptr = nullptr; im.spare = nullptr; im.shares_with = nullptr;
    }
    if (im.ptr) cudaFree(im.ptr);
    if (im.twin) cudaFree(im.twin);
    if (im.staging) cudaFree(im.staging);
    if (im.upload_done) cudaEventDestroy(im.upload_done);
    if (im.staged) cudaEventDestroy(im.staged);
    if (im.staging_free) cudaEventDestroy(im.staging_free);
    if (im.direct_read_done) cudaEventDestroy(im.direct_read_done);
    im = Image();
}
// Orders the compute stream after an asynchronous upload into `im` that it has not consumed yet.
static int consume_upload(vhr_context *ctx, Image *im) {
    if (im && im->upload_pending) {
        VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, im->upload_done, 0));
        im->upload_pending = false;
    }
    return VHR_OK;
}
static int ensure_transfer_queues(vhr_context *ctx) {
    if (!ctx->upload_stream) VHR_CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->upload_stream, cudaStreamNonBlocking));
    if (!ctx->download_stream) VHR_CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->download_stream, cudaStreamNonBlocking));
    if (!ctx->compute_tail) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&ctx->compute_tail, cudaEventDisableTiming));
    return VHR_OK;
}
static Image *find_transient(vhr_context *ctx, const char *name) {
    if (!name) return nullptr;
    auto it = ctx->transient.find(name);
    return it == ctx->transient.end() ? nullptr : &it->second;
}
static int copy_in(vhr_context *ctx, Image *im, const void *host, size_t bytes, const char *what) {
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", what);
    if (!host || bytes != im->bytes) return fail(VHR_ERR_INVALID, "%s: %zu bytes given, image holds %zu", what, bytes, im->bytes);
    if (int rc = consume_upload(ctx, im)) return rc;
    if (int rc = make_writable(ctx, im, true)) return rc;
    VHR_CUDA_CHECK(cudaMemcpyAsync(im->ptr, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return VHR_OK;
}
static int copy_out(vhr_context *ctx, Image *im, void *host, size_t bytes, const char *what) {
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", what);
    if (!host || bytes != im->bytes) return fail(VHR_ERR_INVALID, "%s: %zu bytes given, image holds %zu", what, bytes, im->bytes);
    if (int rc = consume_upload(ctx, im)) return rc;
    VHR_CUDA_CHECK(cudaMemcpyAsync(host, im->ptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return VHR_OK;
}
}  // namespace vhr (anonymous part)

std::string vhr::image_label(vhr_context *ctx, const Image *im) {
    for (auto &kv : ctx->transient)
        if (&kv.second == im) return "'" + kv.first + "'";
    for (size_t s = 0; s < ctx->storage.size(); ++s)
        if (&ctx->storage[s] == im) return "storage image " + std::to_string(s);
    return "unknown image";
}

int vhr::make_writable(vhr_context *ctx, Image *im, bool whole) {
    if (im && im->direct_read_pending) {      // a row read-back straight from the image (vhr_image_download_rows_async) is still in flight
        VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, im->direct_read_done, 0));
        im->direct_read_pending = false;
    }
    if (!im || !im->shares_with) return VHR_OK;
    Image *o = im->shares_with;
    void *sp = im->spare ? im->spare : o->spare;
    void *shared = im->ptr;
    im->ptr = sp;
    im->spare = o->spare = nullptr;
    im->shares_with = o->shares_with = nullptr;
    // everything that read the idle allocation was enqueued before the blit that idled it, i.e. earlier on this stream
    if (!whole) VHR_CUDA_CHECK(cudaMemcpyAsync(im->ptr, shared, im->bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return VHR_OK;
}

namespace vhr {
static int blit(vhr_context *ctx, Image *src, Image *dst, const char *what) {
    if (!src || !dst) return fail(VHR_ERR_INVALID, "%s: unknown image", what);
    // compute_execution_context.cpp:128-129,179-180 assert equal extents; the blit is NEAREST same-size = copy
    if (src->width != dst->width || src->height != dst->height || src->bytes != dst->bytes)
        return fail(VHR_ERR_INVALID, "%s: extents/formats differ (%ux%u fmt %d -> %ux%u fmt %d)", what, src->width,
                    src->height, src->format, dst->width, dst->height, dst->format);
    if (int rc = consume_upload(ctx, src)) return rc;
    if (int rc = consume_upload(ctx, dst)) return rc;
    if (src == dst || (dst->shares_with == src && dst->ptr == src->ptr)) return VHR_OK;      // already the same texels
    if (ctx->part.enabled && ctx->part.world > 1 && src->height == ctx->height) {
        if (int rc = make_writable(ctx, dst, false)) return rc;
        // a rank only ever reads its band and the halo rows around it: copy those (band +- 64 rows)
        const int y0 = std::max(0, ctx->part.band_begin[ctx->part.rank] - 64);
        const int y1 = std::min((int)src->height, ctx->part.band_begin[ctx->part.rank + 1] + 64);
        const size_t row = src->bytes / src->height;
        VHR_CUDA_CHECK(cudaMemcpyAsync((char *)dst->ptr + y0 * row, (const char *)src->ptr + y0 * row, (size_t)(y1 - y0) * row,
                                       cudaMemcpyDeviceToDevice, ctx->stream));
        return VHR_OK;
    }
    if (int rc = make_writable(ctx, dst, true)) return rc;                                   // dst is overwritten: it leaves its old partner
    if (ctx->opt.blit_alias && !src->shares_with && !src->twin && !dst->twin && !src->staging_busy) {
        // copy-free: dst shows src's buffer until one of the two is written again (see Image::shares_with)
        dst->spare = dst->ptr;
        dst->ptr = src->ptr;
        dst->shares_with = src;
        src->shares_with = dst;
        return VHR_OK;
    }
    VHR_CUDA_CHECK(cudaMemcpyAsync(dst->ptr, src->ptr, src->bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return VHR_OK;
}

}  // namespace vhr

using namespace vhr;

#define VHR_NEED_DEVICE(ctx)                                                                                     \
    do {                                                                                                         \
        if ((ctx)->device < 0) return fail(VHR_ERR_CUDA, "%s: context was created with VHR_DEVICE_NONE (no GPU work possible, no CPU fallback)", __func__); \
    } while (0)

extern "C" {

const char *vhr_last_error(void) { return g_error; }

int vhr_context_create(int device, void *cuda_stream, uint32_t width, uint32_t height, vhr_context **out) {
    if (!out) return fail(VHR_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (width == 0 || height == 0) return fail(VHR_ERR_INVALID, "display size %ux%u", width, height);
    if (device == VHR_DEVICE_NONE) {
        // validation-only context: image / storage-slot tables and pass bookkeeping work, every entry point that would
        // touch the GPU fails with VHR_ERR_CUDA. Lets hosts build and check a render graph on a machine without a GPU.
        vhr_context *ctx = new vhr_context();
        ctx->device = VHR_DEVICE_NONE;
        ctx->width = width; ctx->height = height;
        ctx->storage.resize(VHR_MAX_GLOBAL_RESOURCES);
        *out = ctx;
        return VHR_OK;
    }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(VHR_ERR_CUDA, "no CUDA device (%s) — this library has no CPU fallback", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(VHR_ERR_INVALID, "device %d of %d", device, n);
    VHR_CUDA_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    VHR_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(VHR_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    vhr_context *ctx = new vhr_context();
    ctx->device = device;
    ctx->width = width; ctx->height = height;
    ctx->storage.resize(VHR_MAX_GLOBAL_RESOURCES);
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
    } else {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete ctx; return fail(VHR_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
        ctx->own_stream = true;
    }
    ctx->queue[0] = ctx->stream;
    *out = ctx;
    return VHR_OK;
}

void vhr_context_destroy(vhr_context *ctx) {
    if (!ctx) return;
    if (ctx->device < 0) { delete ctx; return; }
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->queue[0]);
    if (ctx->queue[1]) cudaStreamSynchronize(ctx->queue[1]);
    if (ctx->upload_stream) cudaStreamSynchronize(ctx->upload_stream);
    if (ctx->download_stream) cudaStreamSynchronize(ctx->download_stream);
    peer_close_all(ctx);
    for (auto &kv : ctx->transient) free_image(kv.second);
    for (auto &im : ctx->storage) if (im.used) free_image(im);
    free_bvh(ctx);
    free_shadow_scratch(ctx);
    if (ctx->d_vertices) cudaFree(ctx->d_vertices);
    if (ctx->d_indices) cudaFree(ctx->d_indices);
    if (ctx->d_primitives) cudaFree(ctx->d_primitives);
    if (ctx->d_normal_mats) cudaFree(ctx->d_normal_mats);
    if (ctx->d_refl_t) cudaFree(ctx->d_refl_t);
    if (ctx->d_ray_queue) cudaFree(ctx->d_ray_queue);
    for (float4 *q : ctx->d_depth_quads) if (q) cudaFree(q);
    for (float2 *q : ctx->d_depth_tiles) if (q) cudaFree(q);
    for (TextureDesc &t : ctx->textures) if (t.texels) cudaFree((void *)t.texels);
    if (ctx->d_textures) cudaFree(ctx->d_textures);
    if (ctx->d_texel_lut) cudaFree(ctx->d_texel_lut);
    for (cudaEvent_t e : ctx->queries) cudaEventDestroy(e);
    if (ctx->upload_stream) { cudaStreamSynchronize(ctx->upload_stream); cudaStreamDestroy(ctx->upload_stream); }
    if (ctx->download_stream) { cudaStreamSynchronize(ctx->download_stream); cudaStreamDestroy(ctx->download_stream); }
    if (ctx->compute_tail) cudaEventDestroy(ctx->compute_tail);
    for (cudaEvent_t e : ctx->tickets) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->semaphores) if (e) cudaEventDestroy(e);
    if (ctx->queue[1]) cudaStreamDestroy(ctx->queue[1]);
    if (ctx->own_stream) cudaStreamDestroy(ctx->queue[0]);
    delete ctx;
}

int vhr_context_synchronize(vhr_context *ctx) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (ctx->device < 0) return VHR_OK;
    VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->queue[0]));
    if (ctx->queue[1]) VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->queue[1]));
    if (ctx->upload_stream) VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->upload_stream));
    if (ctx->download_stream) VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->download_stream));
    return VHR_OK;
}

int vhr_select_queue(vhr_context *ctx, int queue) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (queue < 0 || queue > 1) return fail(VHR_ERR_INVALID, "queue %d (0 or 1)", queue);
    if (ctx->device < 0) return VHR_OK;      // validation-only context: nothing is recorded
    if (queue == 1 && ctx->part.enabled) return fail(VHR_ERR_STATE, "vhr_select_queue: not available while a partition is set (the peer flag words are ordered on queue 0)");
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (queue == 1 && !ctx->queue[1]) VHR_CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->queue[1], cudaStreamNonBlocking));
    ctx->stream = ctx->queue[queue];
    return VHR_OK;
}

int vhr_queue_signal(vhr_context *ctx, int semaphore) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (semaphore < 0 || semaphore >= VHR_MAX_SEMAPHORES) return fail(VHR_ERR_INVALID, "semaphore %d of %d", semaphore, VHR_MAX_SEMAPHORES);
    if (ctx->device < 0) return VHR_OK;
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (!ctx->semaphores[semaphore]) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&ctx->semaphores[semaphore], cudaEventDisableTiming));
    VHR_CUDA_CHECK(cudaEventRecord(ctx->semaphores[semaphore], ctx->stream));
    ctx->semaphore_signalled[semaphore] = true;
    return VHR_OK;
}

int vhr_queue_wait(vhr_context *ctx, int semaphore) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (semaphore < 0 || semaphore >= VHR_MAX_SEMAPHORES) return fail(VHR_ERR_INVALID, "semaphore %d of %d", semaphore, VHR_MAX_SEMAPHORES);
    if (ctx->device < 0 || !ctx->semaphore_signalled[semaphore]) return VHR_OK;
    VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, ctx->semaphores[semaphore], 0));
    return VHR_OK;
}

int vhr_get_display_size(vhr_context *ctx, uint32_t *width, uint32_t *height) {
    if (!ctx || !width || !height) return fail(VHR_ERR_INVALID, "NULL argument");
    *width = ctx->width; *height = ctx->height;
    return VHR_OK;
}

uint64_t vhr_kernel_launch_count(vhr_context *ctx) { return ctx ? ctx->launches : 0; }

int vhr_update_geometry(vhr_context *ctx, const void *vertices, uint32_t n_vertices, const uint32_t *indices,
                        uint32_t n_indices, const void *primitives, uint32_t n_primitives) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range("UpdateGeometry + BVH build");
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    if ((n_vertices && !vertices) || (n_indices && !indices) || (n_primitives && !primitives))
        return fail(VHR_ERR_INVALID, "NULL geometry array");
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    free_bvh(ctx);
    if (ctx->d_vertices) { cudaFree(ctx->d_vertices); ctx->d_vertices = nullptr; }
    if (ctx->d_indices) { cudaFree(ctx->d_indices); ctx->d_indices = nullptr; }
    if (ctx->d_primitives) { cudaFree(ctx->d_primitives); ctx->d_primitives = nullptr; }
    if (ctx->d_normal_mats) { cudaFree(ctx->d_normal_mats); ctx->d_normal_mats = nullptr; }
    ctx->n_vertices = n_vertices; ctx->n_indices = n_indices; ctx->n_primitives = n_primitives;
    // validate index ranges on the host: an out-of-range index would read outside the vertex buffer on the device
    const Primitive *prims = (const Primitive *)primitives;
    for (uint32_t g = 0; g < n_primitives; ++g) {
        const Primitive &p = prims[g];
        if ((uint64_t)p.index_offset + p.index_count > n_indices)
            return fail(VHR_ERR_INVALID, "primitive %u: indices [%u, +%u) exceed %u", g, p.index_offset, p.index_count, n_indices);
        if (p.vertex_offset > n_vertices) return fail(VHR_ERR_INVALID, "primitive %u: vertex_offset %u exceeds %u", g, p.vertex_offset, n_vertices);
        // a material may only name textures that exist (the reference would sample an unwritten descriptor)
        for (int32_t t : {p.material.base_color_texture, p.material.metallic_roughness_texture, p.material.normal_map})
            if (t >= 0 && ((size_t)t >= ctx->textures.size() || !ctx->textures[t].texels))
                return fail(VHR_ERR_INVALID, "primitive %u: material names texture %d, which has not been uploaded (vhr_upload_texture_from_data)", g, t);
        uint32_t lim = n_vertices - p.vertex_offset;
        for (uint32_t k = 0; k < p.index_count; ++k)
            if (indices[p.index_offset + k] >= lim)
                return fail(VHR_ERR_INVALID, "primitive %u: index %u (+offset %u) exceeds %u vertices", g, indices[p.index_offset + k], p.vertex_offset, n_vertices);
    }
    if (n_vertices) {
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_vertices, (size_t)n_vertices * sizeof(Vertex)));
        VHR_CUDA_CHECK(cudaMemcpyAsync(ctx->d_vertices, vertices, (size_t)n_vertices * sizeof(Vertex), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (n_indices) {
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_indices, (size_t)n_indices * sizeof(uint32_t)));
        VHR_CUDA_CHECK(cudaMemcpyAsync(ctx->d_indices, indices, (size_t)n_indices * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (n_primitives) {
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_primitives, (size_t)n_primitives * sizeof(Primitive)));
        VHR_CUDA_CHECK(cudaMemcpyAsync(ctx->d_primitives, primitives, (size_t)n_primitives * sizeof(Primitive), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (n_primitives) {
        // normal_matrix = glm::inverseTranspose(mat3(transform)) (hybrid_render_path.cpp:45) = cofactor(M) / det(M),
        // evaluated in double like the oracle's G-buffer scaffolding, stored column-major
        std::vector<float> nm((size_t)n_primitives * 9);
        for (uint32_t g = 0; g < n_primitives; ++g) {
            const float *m = prims[g].transform;
            double a00 = m[0], a10 = m[1], a20 = m[2], a01 = m[4], a11 = m[5], a21 = m[6], a02 = m[8], a12 = m[9], a22 = m[10];
            double c00 = a11 * a22 - a21 * a12, c01 = -(a10 * a22 - a20 * a12), c02 = a10 * a21 - a20 * a11;
            double c10 = -(a01 * a22 - a21 * a02), c11 = a00 * a22 - a20 * a02, c12 = -(a00 * a21 - a20 * a01);
            double c20 = a01 * a12 - a11 * a02, c21 = -(a00 * a12 - a10 * a02), c22 = a00 * a11 - a10 * a01;
            double det = a00 * c00 + a01 * c01 + a02 * c02;
            float *o = &nm[(size_t)g * 9];
            o[0] = (float)(c00 / det); o[1] = (float)(c10 / det); o[2] = (float)(c20 / det);
            o[3] = (float)(c01 / det); o[4] = (float)(c11 / det); o[5] = (float)(c21 / det);
            o[6] = (float)(c02 / det); o[7] = (float)(c12 / det); o[8] = (float)(c22 / det);
        }
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_normal_mats, nm.size() * sizeof(float)));
        VHR_CUDA_CHECK(cudaMemcpy(ctx->d_normal_mats, nm.data(), nm.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    int rc = build_bvh(ctx);
    if (rc) return rc;
    // host arrays may be pageable: make sure the async copies have consumed them before returning
    VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    return VHR_OK;
}

int vhr_upload_texture_from_data(vhr_context *ctx, uint32_t width, uint32_t height, const uint8_t *data, int vk_format,
                                 const vhr_sampler_info *sampler_info) {
    if (!ctx || !data) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    if (width == 0 || height == 0 || width > 32768 || height > 32768) return fail(VHR_ERR_INVALID, "texture extent %ux%u", width, height);
    if (vk_format != VHR_FORMAT_R8G8B8A8_UNORM && vk_format != VHR_FORMAT_R8G8B8A8_SRGB)
        return fail(VHR_ERR_INVALID, "texture format %d (R8G8B8A8_UNORM = 37 and R8G8B8A8_SRGB = 43 are what the scene loader uploads)", vk_format);
    // default sampler (resource_manager.cpp:58-69): LINEAR / LINEAR / REPEAT / REPEAT
    vhr_sampler_info si = {VHR_FILTER_LINEAR, VHR_FILTER_LINEAR, VHR_ADDRESS_MODE_REPEAT, VHR_ADDRESS_MODE_REPEAT};
    if (sampler_info) si = *sampler_info;
    if ((si.mag_filter != VHR_FILTER_NEAREST && si.mag_filter != VHR_FILTER_LINEAR) || (si.min_filter != VHR_FILTER_NEAREST && si.min_filter != VHR_FILTER_LINEAR) ||
        si.address_mode_u < 0 || si.address_mode_u > 3 || si.address_mode_v < 0 || si.address_mode_v > 3)
        return fail(VHR_ERR_INVALID, "sampler (mag %d, min %d, u %d, v %d)", si.mag_filter, si.min_filter, si.address_mode_u, si.address_mode_v);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (!ctx->d_textures) {
        ctx->textures.assign(VHR_MAX_GLOBAL_RESOURCES, TextureDesc{nullptr, 0, 0, 0, 0});
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_textures, sizeof(TextureDesc) * VHR_MAX_GLOBAL_RESOURCES));
        VHR_CUDA_CHECK(cudaMemset(ctx->d_textures, 0, sizeof(TextureDesc) * VHR_MAX_GLOBAL_RESOURCES));
        // UNORM8 -> float is c / 255; sRGB8 -> linear is the sRGB EOTF of c / 255 (Khronos Data Format spec 13.3.1), applied per
        // texel BEFORE filtering as Vulkan requires; evaluated in double, rounded once
        float lut[512];
        for (int c = 0; c < 256; ++c) {
            lut[c] = (float)c / 255.0f;
            const double e = (double)c / 255.0;
            lut[256 + c] = (float)(e <= 0.04045 ? e / 12.92 : pow((e + 0.055) / 1.055, 2.4));
        }
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_texel_lut, sizeof(lut)));
        VHR_CUDA_CHECK(cudaMemcpy(ctx->d_texel_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
    }
    int slot = -1;                                   // first free slot, resource_manager.cpp:821-824
    for (int i = 0; i < VHR_MAX_GLOBAL_RESOURCES; ++i)
        if (!ctx->textures[i].texels) { slot = i; break; }
    if (slot < 0) return fail(VHR_ERR_EXHAUSTED, "no free texture slot (%d in use)", VHR_MAX_GLOBAL_RESOURCES);
    const size_t bytes = (size_t)width * height * 4;
    void *texels = nullptr;
    VHR_CUDA_CHECK(cudaMalloc(&texels, bytes));
    cudaError_t e = cudaMemcpy(texels, data, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(texels); return fail(VHR_ERR_CUDA, "texture upload: %s", cudaGetErrorString(e)); }
    TextureDesc d;
    d.texels = (const uint32_t *)texels; d.width = width; d.height = height; d.pad = 0;
    d.flags = (vk_format == VHR_FORMAT_R8G8B8A8_SRGB ? 1u : 0u) | (si.mag_filter == VHR_FILTER_LINEAR ? 2u : 0u) | (si.min_filter == VHR_FILTER_LINEAR ? 4u : 0u) |
              ((uint32_t)si.address_mode_u << 4) | ((uint32_t)si.address_mode_v << 6);
    ctx->textures[slot] = d;
    VHR_CUDA_CHECK(cudaMemcpy(ctx->d_textures + slot, &d, sizeof(d), cudaMemcpyHostToDevice));
    return slot;
}

int vhr_destroy_textures(vhr_context *ctx) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (ctx->device < 0 || !ctx->d_textures) return VHR_OK;
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    for (TextureDesc &t : ctx->textures)
        if (t.texels) { cudaFree((void *)t.texels); t = TextureDesc{nullptr, 0, 0, 0, 0}; }
    VHR_CUDA_CHECK(cudaMemset(ctx->d_textures, 0, sizeof(TextureDesc) * VHR_MAX_GLOBAL_RESOURCES));
    return VHR_OK;
}

int vhr_update_per_frame_ubo(vhr_context *ctx, const void *per_frame_data, size_t size) {
    if (ctx) ctx->epoch++;
    if (!ctx || !per_frame_data) return fail(VHR_ERR_INVALID, "NULL argument");
    if (size != sizeof(PerFrameData)) return fail(VHR_ERR_INVALID, "PerFrameData is %zu bytes, got %zu", sizeof(PerFrameData), size);
    memcpy(&ctx->pfd, per_frame_data, sizeof(PerFrameData));
    ctx->pfd_set = true;
    return VHR_OK;
}

int vhr_upload_new_storage_image(vhr_context *ctx, uint32_t width, uint32_t height, int vk_format) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (ctx->device >= 0) VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    for (int i = 0; i < VHR_MAX_GLOBAL_RESOURCES; ++i) {
        if (!ctx->storage[i].used) {
            int rc = alloc_image(ctx, ctx->storage[i], width, height, vk_format);
            return rc ? rc : i;
        }
    }
    return fail(VHR_ERR_EXHAUSTED, "No free storage image slots left!");
}

int vhr_destroy_storage_image(vhr_context *ctx, int slot) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    Image *im = storage_slot(ctx, slot);
    if (!im) return fail(VHR_ERR_INVALID, "storage image %d does not exist", slot);
    if (ctx->device >= 0) VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    free_image(*im);
    return VHR_OK;
}

int vhr_actualize_image(vhr_context *ctx, const char *name, uint32_t width, uint32_t height, int vk_format) {
    if (!ctx || !name) return fail(VHR_ERR_INVALID, "NULL argument");
    if (ctx->device >= 0) VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (width == 0 && height == 0) { width = ctx->width; height = ctx->height; }
    Image *im = find_transient(ctx, name);
    if (im) {
        if (im->width != width || im->height != height || im->format != vk_format)
            return fail(VHR_ERR_INVALID, "image '%s' re-declared as %ux%u fmt %d (is %ux%u fmt %d)", name, width, height,
                        vk_format, im->width, im->height, im->format);
        return VHR_OK;
    }
    Image fresh;
    int rc = alloc_image(ctx, fresh, width, height, vk_format);
    if (rc) return rc;
    ctx->transient[name] = fresh;
    return VHR_OK;
}

int vhr_destroy_transient_resources(vhr_context *ctx) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (ctx->device >= 0) VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    for (auto &kv : ctx->transient) free_image(kv.second);
    ctx->transient.clear();
    ctx->n_bound = 0;
    return VHR_OK;
}

int vhr_image_upload(vhr_context *ctx, const char *name, const void *host, size_t bytes) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return copy_in(ctx, find_transient(ctx, name), host, bytes, name ? name : "(null)");
}
int vhr_image_download(vhr_context *ctx, const char *name, void *host, size_t bytes) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return copy_out(ctx, find_transient(ctx, name), host, bytes, name ? name : "(null)");
}
int vhr_storage_image_upload(vhr_context *ctx, int slot, const void *host, size_t bytes) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return copy_in(ctx, storage_slot(ctx, slot), host, bytes, "storage image");
}
int vhr_storage_image_download(vhr_context *ctx, int slot, void *host, size_t bytes) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return copy_out(ctx, storage_slot(ctx, slot), host, bytes, "storage image");
}
int vhr_image_upload_async(vhr_context *ctx, const char *name, const void *host, size_t bytes) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    Image *im = find_transient(ctx, name);
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", name ? name : "(null)");
    if (!host || bytes != im->bytes) return fail(VHR_ERR_INVALID, "%s: %zu bytes given, image holds %zu", name, bytes, im->bytes);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (int rc = ensure_transfer_queues(ctx)) return rc;
    if (int rc = make_writable(ctx, im, true)) return rc;
    if (!im->upload_done) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&im->upload_done, cudaEventDisableTiming));
    // the copy may only start once every pass enqueued so far (the image's last readers) has finished
    VHR_CUDA_CHECK(cudaEventRecord(ctx->compute_tail, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->upload_stream, ctx->compute_tail, 0));
    VHR_CUDA_CHECK(cudaMemcpyAsync(im->ptr, host, bytes, cudaMemcpyHostToDevice, ctx->upload_stream));
    VHR_CUDA_CHECK(cudaEventRecord(im->upload_done, ctx->upload_stream));
    im->upload_pending = true;
    return VHR_OK;
}

int vhr_image_download_async(vhr_context *ctx, const char *name, void *host, size_t bytes, uint32_t *ticket) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    Image *im = find_transient(ctx, name);
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", name ? name : "(null)");
    if (!host || !ticket || bytes != im->bytes) return fail(VHR_ERR_INVALID, "%s: %zu bytes given, image holds %zu", name, bytes, im->bytes);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (int rc = ensure_transfer_queues(ctx)) return rc;
    if (int rc = consume_upload(ctx, im)) return rc;
    if (!im->staging) {
        VHR_CUDA_CHECK(cudaMalloc(&im->staging, im->bytes));
        VHR_CUDA_CHECK(cudaEventCreateWithFlags(&im->staged, cudaEventDisableTiming));
        VHR_CUDA_CHECK(cudaEventCreateWithFlags(&im->staging_free, cudaEventDisableTiming));
    }
    // snapshot on the compute stream (a device-to-device copy at HBM speed), so later passes may overwrite the image
    // while the PCIe copy is still in flight; the snapshot itself is reused only after its previous read-back
    if (im->staging_busy) VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, im->staging_free, 0));
    VHR_CUDA_CHECK(cudaMemcpyAsync(im->staging, im->ptr, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    VHR_CUDA_CHECK(cudaEventRecord(im->staged, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->download_stream, im->staged, 0));
    VHR_CUDA_CHECK(cudaMemcpyAsync(host, im->staging, bytes, cudaMemcpyDeviceToHost, ctx->download_stream));
    VHR_CUDA_CHECK(cudaEventRecord(im->staging_free, ctx->download_stream));
    im->staging_busy = true;
    if (ctx->tickets.empty()) {
        ctx->tickets.resize(64);
        for (auto &e : ctx->tickets) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const uint32_t t = ctx->next_ticket++;
    VHR_CUDA_CHECK(cudaEventRecord(ctx->tickets[t % ctx->tickets.size()], ctx->download_stream));
    *ticket = t;
    return VHR_OK;
}

int vhr_wait_download(vhr_context *ctx, uint32_t ticket) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    if (ticket >= ctx->next_ticket) return fail(VHR_ERR_INVALID, "download ticket %u was never issued", ticket);
    if (ctx->next_ticket - ticket > ctx->tickets.size()) return VHR_OK;   // recycled: that download finished long ago
    VHR_CUDA_CHECK(cudaEventSynchronize(ctx->tickets[ticket % ctx->tickets.size()]));
    return VHR_OK;
}

void *vhr_image_device_ptr(vhr_context *ctx, const char *name, uint32_t *width, uint32_t *height, int *vk_format) {
    Image *im = ctx ? find_transient(ctx, name) : nullptr;
    if (!im) return nullptr;
    if (width) *width = im->width;
    if (height) *height = im->height;
    if (vk_format) *vk_format = im->format;
    return im->ptr;
}
void *vhr_storage_image_device_ptr(vhr_context *ctx, int slot, uint32_t *width, uint32_t *height, int *vk_format) {
    Image *im = ctx ? storage_slot(ctx, slot) : nullptr;
    if (!im) return nullptr;
    if (width) *width = im->width;
    if (height) *height = im->height;
    if (vk_format) *vk_format = im->format;
    return im->ptr;
}

int vhr_bind_pass_images(vhr_context *ctx, const char *const *names_by_binding, uint32_t count) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (count > VHR_MAX_PASS_BINDINGS) return fail(VHR_ERR_INVALID, "%u bindings (max %d)", count, VHR_MAX_PASS_BINDINGS);
    for (uint32_t i = 0; i < count; ++i) {
        Image *im = names_by_binding ? find_transient(ctx, names_by_binding[i]) : nullptr;
        if (!im) return fail(VHR_ERR_INVALID, "binding %u: unknown image '%s'", i, (names_by_binding && names_by_binding[i]) ? names_by_binding[i] : "(null)");
        if (ctx->device >= 0)
            if (int rc = consume_upload(ctx, im)) return rc;
        ctx->bound[i] = im;
    }
    ctx->n_bound = count;
    return VHR_OK;
}

int vhr_dispatch(vhr_context *ctx, const char *shader_path, uint32_t x_groups, uint32_t y_groups, uint32_t z_groups,
                 const void *push_constants, size_t push_constants_size) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range(shader_path);
    if (!ctx || !shader_path) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    if (!ctx->pfd_set) return fail(VHR_ERR_STATE, "vhr_update_per_frame_ubo has not been called");
    if (z_groups != 1) return fail(VHR_ERR_INVALID, "z_groups = %u (the hot-path kernels are 2D)", z_groups);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    const bool is_temporal = !strcmp(shader_path, "hybrid_render_path/svgf.comp");
    const bool is_atrous = !strcmp(shader_path, "hybrid_render_path/svgf_atrous_filter.comp");
    if (is_temporal || is_atrous) {
        // compute_execution_context.h:23: assert(sizeof(T) == pipeline.push_constant_description.size)
        if (!push_constants || push_constants_size != sizeof(SVGFPushConstants))
            return fail(VHR_ERR_INVALID, "%s: push constants are %zu bytes, got %zu", shader_path, sizeof(SVGFPushConstants), push_constants_size);
        SVGFPushConstants pc;
        memcpy(&pc, push_constants, sizeof(pc));
        return is_temporal ? launch_svgf_temporal(ctx, x_groups, y_groups, pc) : launch_svgf_atrous(ctx, x_groups, y_groups, pc);
    }
    if (!strcmp(shader_path, "hybrid_render_path/ssao.comp")) {
        // SURVEY Q15: the reference never pushes the radius to this kernel; intent 0.75 (hybrid_render_path.cpp:139-141)
        float radius = 0.75f;
        if (push_constants) {
            if (push_constants_size != sizeof(SSAOPushConstants))
                return fail(VHR_ERR_INVALID, "%s: push constants are %zu bytes, got %zu", shader_path, sizeof(SSAOPushConstants), push_constants_size);
            memcpy(&radius, push_constants, sizeof(float));
        }
        return launch_ssao(ctx, x_groups, y_groups, radius);
    }
    if (!strcmp(shader_path, "hybrid_render_path/ssao_blur.comp")) {
        // the reference pushes SSAOPushConstants here although the shader has no push-constant block (Q15): accepted, ignored
        if (push_constants && push_constants_size != sizeof(SSAOPushConstants))
            return fail(VHR_ERR_INVALID, "%s: push constants are %zu bytes, got %zu", shader_path, sizeof(SSAOPushConstants), push_constants_size);
        return launch_ssao_blur(ctx, x_groups, y_groups);
    }
    if (!strcmp(shader_path, "hybrid_render_path/ssr.comp")) {
        if (!push_constants || push_constants_size != sizeof(SSRPushConstants))
            return fail(VHR_ERR_INVALID, "%s: push constants are %zu bytes, got %zu", shader_path, sizeof(SSRPushConstants), push_constants_size);
        SSRPushConstants pc;
        memcpy(&pc, push_constants, sizeof(pc));
        return launch_ssr(ctx, x_groups, y_groups, pc);
    }
    return fail(VHR_ERR_INVALID, "unknown compute kernel '%s'", shader_path);
}

int vhr_trace_rays(vhr_context *ctx, const char *pipeline_name, uint32_t width, uint32_t height) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range(pipeline_name);
    if (!ctx || !pipeline_name) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    const bool hybrid = !strcmp(pipeline_name, "Raytrace Pipeline"), full = !strcmp(pipeline_name, "Raytracing Pipeline");
    if (!hybrid && !full) return fail(VHR_ERR_INVALID, "unknown ray-tracing pipeline '%s'", pipeline_name);
    if (!ctx->pfd_set) return fail(VHR_ERR_STATE, "vhr_update_per_frame_ubo has not been called");
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    return hybrid ? launch_trace_rays(ctx, width, height) : launch_raytraced(ctx, width, height);
}

int vhr_draw(vhr_context *ctx, const char *fragment_shader, const int32_t *specialization_constants, uint32_t n_constants,
             uint32_t vertex_count, uint32_t instance_count, uint32_t first_vertex, uint32_t first_instance) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range(fragment_shader);
    if (!ctx || !fragment_shader) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    if (!ctx->pfd_set) return fail(VHR_ERR_STATE, "vhr_update_per_frame_ubo has not been called");
    const bool present = !strcmp(fragment_shader, "raytraced_render_path/composition.frag");
    if (!present && strcmp(fragment_shader, "hybrid_render_path/composition.frag"))
        return fail(VHR_ERR_INVALID, "vhr_draw: no kernel for fragment shader '%s' (only the composition passes are CUDA kernels)", fragment_shader);
    if (present) {
        if (vertex_count != 3 || instance_count != 1 || first_vertex != 0 || first_instance != 0)
            return fail(VHR_ERR_INVALID, "vhr_draw: composition is Draw(3, 1, 0, 0), got (%u, %u, %u, %u)", vertex_count, instance_count, first_vertex, first_instance);
        VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
        return launch_present(ctx);
    }
    if (vertex_count != 3 || instance_count != 1 || first_vertex != 0 || first_instance != 0)
        return fail(VHR_ERR_INVALID, "vhr_draw: composition is Draw(3, 1, 0, 0), got (%u, %u, %u, %u)", vertex_count, instance_count, first_vertex, first_instance);
    if (!specialization_constants || n_constants != 3)
        return fail(VHR_ERR_INVALID, "vhr_draw: composition.frag takes 3 specialization constants, got %u", n_constants);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    return launch_composition(ctx, specialization_constants[0], specialization_constants[1], specialization_constants[2]);
}

int vhr_gbuffer_pass(vhr_context *ctx, uint32_t width, uint32_t height) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range("G-Buffer Pass (primary rays)");
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    if (!ctx->pfd_set) return fail(VHR_ERR_STATE, "vhr_update_per_frame_ubo has not been called");
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    return launch_gbuffer(ctx, width, height);
}

int vhr_shadow_map_pass(vhr_context *ctx) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range("Shadow Map Pass");
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    if (!ctx->pfd_set) return fail(VHR_ERR_STATE, "vhr_update_per_frame_ubo has not been called");
    if (!ctx->d_primitives) return fail(VHR_ERR_STATE, "Shadow Map Pass: no geometry (vhr_update_geometry)");
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    return launch_shadow_map(ctx);
}

int vhr_trace_explicit(vhr_context *ctx, const float *rays, uint32_t n, int any_hit, float *out_t, uint32_t *out_ids,
                       float *out_uv) {
    if (!ctx || (n && (!rays || !out_t))) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    return launch_trace_explicit(ctx, rays, n, any_hit, out_t, out_ids, out_uv);
}

int vhr_blit_storage_to_transient(vhr_context *ctx, int src_slot, const char *dst_name) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range("BlitImageStorageToTransient");
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return blit(ctx, storage_slot(ctx, src_slot), find_transient(ctx, dst_name), "BlitImageStorageToTransient");
}
int vhr_blit_transient_to_storage(vhr_context *ctx, const char *src_name, int dst_slot) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range("BlitImageTransientToStorage");
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return blit(ctx, find_transient(ctx, src_name), storage_slot(ctx, dst_slot), "BlitImageTransientToStorage");
}
int vhr_blit_storage_to_storage(vhr_context *ctx, int src_slot, int dst_slot) {
    if (ctx) ctx->epoch++;
    NvtxRange nvtx_range("BlitImageStorageToStorage");
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    return blit(ctx, storage_slot(ctx, src_slot), storage_slot(ctx, dst_slot), "BlitImageStorageToStorage");
}

int vhr_cmd_begin_debug_label(vhr_context *ctx, const char *label) {
    if (!ctx || !label) return fail(VHR_ERR_INVALID, "NULL argument");
    nvtxRangePushA(label);
    ctx->debug_label_depth++;
    return VHR_OK;
}
int vhr_cmd_end_debug_label(vhr_context *ctx) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (ctx->debug_label_depth == 0) return fail(VHR_ERR_STATE, "vhr_cmd_end_debug_label without a matching begin");
    nvtxRangePop();
    ctx->debug_label_depth--;
    return VHR_OK;
}

// Rows [y0, y1) of an image, on the transfer queues (the row-band partition moves only a band of the G-buffer up and a band of the
// result down). Same ordering rules as the whole-image calls above.
int vhr_image_upload_rows_async(vhr_context *ctx, const char *name, const void *host_rows, uint32_t y0, uint32_t y1) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    Image *im = find_transient(ctx, name);
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", name ? name : "(null)");
    if (!host_rows || y0 >= y1 || y1 > im->height) return fail(VHR_ERR_INVALID, "%s: rows [%u, %u) of %u", name, y0, y1, im->height);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (int rc = ensure_transfer_queues(ctx)) return rc;
    if (int rc = make_writable(ctx, im, false)) return rc;
    if (!im->upload_done) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&im->upload_done, cudaEventDisableTiming));
    const size_t row = im->bytes / im->height;
    VHR_CUDA_CHECK(cudaEventRecord(ctx->compute_tail, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->upload_stream, ctx->compute_tail, 0));
    VHR_CUDA_CHECK(cudaMemcpyAsync((char *)im->ptr + (size_t)y0 * row, host_rows, (size_t)(y1 - y0) * row, cudaMemcpyHostToDevice, ctx->upload_stream));
    VHR_CUDA_CHECK(cudaEventRecord(im->upload_done, ctx->upload_stream));
    im->upload_pending = true;
    return VHR_OK;
}
// Every `stride_rows`-th block of `block_rows` rows starting at row `first_row`, `n_blocks` of them, from a host image of the same row
// pitch (host_image points at row 0 of the FULL host image): the rows a rank of the fused partition ray-traces (8-row blocks dealt
// round-robin). One strided DMA (cudaMemcpy2DAsync) instead of n_blocks copies.
int vhr_image_upload_blocks_async(vhr_context *ctx, const char *name, const void *host_image, uint32_t first_row, uint32_t block_rows,
                                  uint32_t stride_rows, uint32_t n_blocks) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    Image *im = find_transient(ctx, name);
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", name ? name : "(null)");
    if (!host_image || block_rows == 0 || stride_rows < block_rows || n_blocks == 0 ||
        (uint64_t)first_row + (uint64_t)(n_blocks - 1) * stride_rows + block_rows > im->height)
        return fail(VHR_ERR_INVALID, "%s: blocks of %u rows every %u rows from row %u x %u exceed %u rows", name, block_rows, stride_rows, first_row, n_blocks, im->height);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (int rc = ensure_transfer_queues(ctx)) return rc;
    if (int rc = make_writable(ctx, im, false)) return rc;
    if (!im->upload_done) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&im->upload_done, cudaEventDisableTiming));
    const size_t row = im->bytes / im->height;
    VHR_CUDA_CHECK(cudaEventRecord(ctx->compute_tail, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->upload_stream, ctx->compute_tail, 0));
    VHR_CUDA_CHECK(cudaMemcpy2DAsync((char *)im->ptr + (size_t)first_row * row, (size_t)stride_rows * row, (const char *)host_image + (size_t)first_row * row,
                                     (size_t)stride_rows * row, (size_t)block_rows * row, n_blocks, cudaMemcpyHostToDevice, ctx->upload_stream));
    VHR_CUDA_CHECK(cudaEventRecord(im->upload_done, ctx->upload_stream));
    im->upload_pending = true;
    return VHR_OK;
}
// Reads rows [y0, y1) straight from the image (no device-side snapshot): the caller must not enqueue anything that rewrites the image
// before vhr_wait_download(ticket) — true for an image that is only written once per frame when the host waits for frame k's read-back
// before it records frame k+1's writer, which is what a frame loop with one frame of latency does.
int vhr_image_download_rows_async(vhr_context *ctx, const char *name, void *host_rows, uint32_t y0, uint32_t y1, uint32_t *ticket) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    VHR_NEED_DEVICE(ctx);
    Image *im = find_transient(ctx, name);
    if (!im) return fail(VHR_ERR_INVALID, "%s: unknown image", name ? name : "(null)");
    if (!host_rows || !ticket || y0 >= y1 || y1 > im->height) return fail(VHR_ERR_INVALID, "%s: rows [%u, %u) of %u", name, y0, y1, im->height);
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (int rc = ensure_transfer_queues(ctx)) return rc;
    if (int rc = consume_upload(ctx, im)) return rc;
    const size_t row = im->bytes / im->height;
    VHR_CUDA_CHECK(cudaEventRecord(ctx->compute_tail, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamWaitEvent(ctx->download_stream, ctx->compute_tail, 0));
    VHR_CUDA_CHECK(cudaMemcpyAsync(host_rows, (const char *)im->ptr + (size_t)y0 * row, (size_t)(y1 - y0) * row, cudaMemcpyDeviceToHost, ctx->download_stream));
    if (ctx->tickets.empty()) {
        ctx->tickets.resize(64);
        for (auto &e : ctx->tickets) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const uint32_t t = ctx->next_ticket++;
    VHR_CUDA_CHECK(cudaEventRecord(ctx->tickets[t % ctx->tickets.size()], ctx->download_stream));
    // the next WRITER of this image on the compute stream must come after this read (make_writable, which every writer calls, waits for
    // it); everything else enqueued on the compute stream runs under the copy
    if (!im->direct_read_done) VHR_CUDA_CHECK(cudaEventCreateWithFlags(&im->direct_read_done, cudaEventDisableTiming));
    VHR_CUDA_CHECK(cudaEventRecord(im->direct_read_done, ctx->download_stream));
    im->direct_read_pending = true;
    *ticket = t;
    return VHR_OK;
}

int vhr_create_query_pool(vhr_context *ctx, uint32_t count) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    if (ctx->device < 0) return VHR_OK;
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    for (cudaEvent_t e : ctx->queries) cudaEventDestroy(e);
    ctx->queries.assign(count, nullptr);
    for (uint32_t i = 0; i < count; ++i) VHR_CUDA_CHECK(cudaEventCreate(&ctx->queries[i]));
    return VHR_OK;
}
int vhr_write_timestamp(vhr_context *ctx, uint32_t query) {
    if (!ctx || query >= ctx->queries.size()) return fail(VHR_ERR_INVALID, "timestamp query %u out of range", query);
    VHR_NEED_DEVICE(ctx);
    VHR_CUDA_CHECK(cudaEventRecord(ctx->queries[query], ctx->stream));
    return VHR_OK;
}
int vhr_get_query_elapsed_ms(vhr_context *ctx, uint32_t first, uint32_t last, double *out_ms) {
    if (!ctx || !out_ms) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    if (first >= ctx->queries.size() || last >= ctx->queries.size())
        return fail(VHR_ERR_INVALID, "timestamp query range [%u, %u] invalid", first, last);
    VHR_CUDA_CHECK(cudaEventSynchronize(ctx->queries[last]));
    float ms = 0.0f;
    VHR_CUDA_CHECK(cudaEventElapsedTime(&ms, ctx->queries[first], ctx->queries[last]));
    *out_ms = ms;
    return VHR_OK;
}

int vhr_set_option(vhr_context *ctx, int option, int64_t value) {
    if (ctx) ctx->epoch++;
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    switch (option) {
        case VHR_OPT_AO_SPP:
            // 0 would make the kernel average zero samples (0 / 0 = NaN into the RG16F image); VHR_OPT_TRACE_AO = 0 switches AO off
            if (value < 1 || value > 64) return fail(VHR_ERR_INVALID, "ao_spp %lld out of [1, 64]", (long long)value);
            ctx->opt.ao_spp = (int)value; return VHR_OK;
        case VHR_OPT_TRACE_SHADOWS: ctx->opt.trace_shadows = value != 0; return VHR_OK;
        case VHR_OPT_TRACE_AO: ctx->opt.trace_ao = value != 0; return VHR_OK;
        case VHR_OPT_TRACE_REFLECTIONS: ctx->opt.trace_reflections = value != 0; return VHR_OK;
        case VHR_OPT_ROW_BEGIN: ctx->opt.row_begin = (int)value; return VHR_OK;
        case VHR_OPT_ROW_END: ctx->opt.row_end = (int)value; return VHR_OK;
        case VHR_OPT_SVGF_FUSED: ctx->opt.svgf_fused = value != 0; return VHR_OK;
        case VHR_OPT_BLIT_ALIAS: ctx->opt.blit_alias = value != 0; return VHR_OK;
        case VHR_OPT_ATROUS_VARIANT:
            if (value < 0 || value > 3) return fail(VHR_ERR_INVALID, "atrous variant %lld", (long long)value);
            ctx->opt.atrous_variant = (int)value; return VHR_OK;
        case VHR_OPT_RAYTRACED_ALPHA_TEST: ctx->opt.raytraced_alpha_test = value != 0; return VHR_OK;
        case VHR_OPT_OUTPUT_RANK:
            if (value < -1 || value >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "output rank %lld out of [-1, %d]", (long long)value, VHR_MAX_RANKS - 1);
            ctx->opt.output_rank = (int)value; return VHR_OK;
        case VHR_OPT_RAYGEN_VARIANT:
            if (value < 0 || value > 15 || value == 5) return fail(VHR_ERR_INVALID, "raygen variant %lld", (long long)value);
            ctx->opt.raygen_variant = (int)value; return VHR_OK;
        case VHR_OPT_DEBUG_REFLECTION_T:
            ctx->opt.debug_refl_t = value != 0;
            if (ctx->device < 0) return VHR_OK;
            if (ctx->opt.debug_refl_t && !ctx->d_refl_t) {
                VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
                VHR_CUDA_CHECK(cudaMalloc(&ctx->d_refl_t, (size_t)ctx->width * ctx->height * sizeof(float)));
            } else if (!ctx->opt.debug_refl_t && ctx->d_refl_t) {
                cudaStreamSynchronize(ctx->stream);
                cudaFree(ctx->d_refl_t);
                ctx->d_refl_t = nullptr;
            }
            return VHR_OK;
    }
    return fail(VHR_ERR_INVALID, "unknown option %d", option);
}

int64_t vhr_get_option(vhr_context *ctx, int option) {
    if (!ctx) return -1;
    switch (option) {
        case VHR_OPT_AO_SPP: return ctx->opt.ao_spp;
        case VHR_OPT_TRACE_SHADOWS: return ctx->opt.trace_shadows;
        case VHR_OPT_TRACE_AO: return ctx->opt.trace_ao;
        case VHR_OPT_TRACE_REFLECTIONS: return ctx->opt.trace_reflections;
        case VHR_OPT_ROW_BEGIN: return ctx->opt.row_begin;
        case VHR_OPT_ROW_END: return ctx->opt.row_end;
        case VHR_OPT_SVGF_FUSED: return ctx->opt.svgf_fused;
        case VHR_OPT_BLIT_ALIAS: return ctx->opt.blit_alias;
        case VHR_OPT_ATROUS_VARIANT: return ctx->opt.atrous_variant;
        case VHR_OPT_DEBUG_REFLECTION_T: return ctx->opt.debug_refl_t;
        case VHR_OPT_RAYGEN_VARIANT: return ctx->opt.raygen_variant;
        case VHR_OPT_RAYTRACED_ALPHA_TEST: return ctx->opt.raytraced_alpha_test;
        case VHR_OPT_OUTPUT_RANK: return ctx->opt.output_rank;
    }
    return -1;
}

int vhr_debug_download_reflection_t(vhr_context *ctx, float *host, size_t bytes) {
    if (!ctx || !host) return fail(VHR_ERR_INVALID, "NULL argument");
    VHR_NEED_DEVICE(ctx);
    if (!ctx->d_refl_t) return fail(VHR_ERR_STATE, "VHR_OPT_DEBUG_REFLECTION_T is not enabled");
    size_t need = (size_t)ctx->width * ctx->height * sizeof(float);
    if (bytes != need) return fail(VHR_ERR_INVALID, "reflection-t image is %zu bytes, got %zu", need, bytes);
    VHR_CUDA_CHECK(cudaMemcpyAsync(host, ctx->d_refl_t, need, cudaMemcpyDeviceToHost, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    return VHR_OK;
}

int vhr_debug_shade_hits(vhr_context *ctx, int kind, const vhr_shade_record *records, uint32_t n, uint32_t *out) {
    if (!ctx || (n && (!records || !out))) return fail(VHR_ERR_INVALID, "NULL argument");
    if (kind < VHR_SHADE_TEXTURE || kind > VHR_SHADE_ANYHIT_ALPHA) return fail(VHR_ERR_INVALID, "vhr_debug_shade_hits: kind %d", kind);
    VHR_NEED_DEVICE(ctx);
    if (!ctx->pfd_set) return fail(VHR_ERR_STATE, "vhr_update_per_frame_ubo has not been called");
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (kind == VHR_SHADE_TEXTURE) {
        for (uint32_t i = 0; i < n; ++i)
            if (records[i].g >= ctx->textures.size() || !ctx->textures[records[i].g].texels)
                return fail(VHR_ERR_INVALID, "vhr_debug_shade_hits: record %u names texture slot %u, which holds no texture", i, records[i].g);
    } else {
        if (!ctx->d_primitives) return fail(VHR_ERR_STATE, "vhr_debug_shade_hits: no geometry (vhr_update_geometry)");
        std::vector<Primitive> prims(ctx->n_primitives);
        VHR_CUDA_CHECK(cudaMemcpyAsync(prims.data(), ctx->d_primitives, prims.size() * sizeof(Primitive), cudaMemcpyDeviceToHost, ctx->stream));
        VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        for (uint32_t i = 0; i < n; ++i)
            if (records[i].g >= ctx->n_primitives || records[i].pid >= prims[records[i].g].index_count / 3)
                return fail(VHR_ERR_INVALID, "vhr_debug_shade_hits: record %u names triangle %u of geometry %u (%u geometries)", i, records[i].pid,
                            records[i].g, ctx->n_primitives);
    }
    return launch_shade_hits(ctx, kind, records, n, out);
}

int vhr_get_bvh_stats(vhr_context *ctx, vhr_bvh_stats *out) {
    if (!ctx || !out) return fail(VHR_ERR_INVALID, "NULL argument");
    *out = ctx->bvh.stats;
    return VHR_OK;
}

}  // extern "C"
