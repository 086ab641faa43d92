/* vhr_b200.h — C-ABI of the B200-native ray-traced lighting + SVGF/SSAO chain.
 *
 * Drop-in boundary for the hybrid render path of RMichelsen/VulkanHybridRenderer: every entry point replaces one
 * call the reference's RenderGraph / ResourceManager / execution contexts make into the Vulkan driver for this path.
 * Citations are relative to the reference tree. Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions
 *   - every function returns 0 on success, a negative vhr_status otherwise (the reference asserts / prints instead:
 *     src/rendering_backend/vulkan_common.h:4-7); vhr_last_error() holds the message of the last failure on the
 *     calling thread.
 *   - one context = one GPU + one CUDA stream; all work is enqueued on that stream in call order (the reference
 *     records everything into one command buffer on one queue, src/rendering_backend/renderer.cpp:135). A context is
 *     not thread-safe, like the reference's single-threaded recording (src/main.cpp:111-127).
 *   - images are linear, dense row-major device buffers in the reference's texel formats; row 0 is NDC y = -1.
 *   - there is NO CPU fallback: every compute entry point fails with VHR_ERR_CUDA when no sm_100 device is present.
 */
#ifndef VHR_B200_H
#define VHR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vhr_context vhr_context;

typedef enum vhr_status {
    VHR_OK = 0,
    VHR_ERR_INVALID = -1,      /* bad argument / unknown name / size mismatch (reference: assert) */
    VHR_ERR_CUDA = -2,         /* CUDA runtime failure or no usable device */
    VHR_ERR_EXHAUSTED = -3,    /* no free storage-image slot (reference: resource_manager.cpp:876-877) */
    VHR_ERR_STATE = -4         /* call order violated (e.g. trace before geometry upload) */
} vhr_status;

/* VkFormat values accepted for images (src/render_paths/hybrid_render_path.cpp:16-19,109-110,247-261). */
enum {
    VHR_FORMAT_R8G8B8A8_UNORM = 37,  /* material textures: metallic-roughness, normal maps (scene_loader.cpp:258-272) */
    VHR_FORMAT_R8G8B8A8_SRGB = 43,   /* material textures: base colour (scene_loader.cpp:249-252) */
    VHR_FORMAT_B8G8R8A8_UNORM = 44,
    VHR_FORMAT_B8G8R8A8_SRGB = 50,   /* the swapchain format RENDER_OUTPUT has in the reference (vulkan_context.cpp:331) */
    VHR_FORMAT_R16G16_SFLOAT = 83,
    VHR_FORMAT_R16G16B16A16_SFLOAT = 97,
    VHR_FORMAT_D32_SFLOAT = 126
};

/* device index for a validation-only context: image/slot tables and pass bookkeeping work (so a host can build and
 * sanity-check its render graph on a machine without a GPU); every entry point that needs the GPU fails with
 * VHR_ERR_CUDA. This is not a CPU fallback: nothing is ever computed on the host. */
#define VHR_DEVICE_NONE (-1)

#define VHR_MAX_GLOBAL_RESOURCES 2048   /* src/rendering_backend/resource_manager.h:13 */
#define VHR_MAX_PASS_BINDINGS 16
#define VHR_MAX_RANKS 8                 /* GPUs of one NVSwitch box a frame can be partitioned over */
#define VHR_IPC_HANDLE_BYTES 64         /* sizeof(cudaIpcMemHandle_t) */

/* ---- context (replaces VulkanContext device/queue creation, src/rendering_backend/vulkan_context.cpp:44) -------- */

/* `cuda_stream` may be NULL (the context creates its own non-blocking stream) or an existing cudaStream_t / CUstream
 * of `device` (e.g. torch.cuda.current_stream().cuda_stream) so callers can time the passes with their own events.
 * width/height = the swapchain extent every "swapchain-sized" (0,0) transient image takes
 * (src/render_graph/render_graph.cpp:962-966). */
int vhr_context_create(int device, void *cuda_stream, uint32_t width, uint32_t height, vhr_context **out);
void vhr_context_destroy(vhr_context *ctx);
const char *vhr_last_error(void);
/* Blocks until everything enqueued on the context's stream has finished, a deferred a-trous dispatch included (vhr_dispatch)
 * (reference: vkWaitForFences, renderer.cpp:107). */
int vhr_context_synchronize(vhr_context *ctx);
/* ComputeExecutionContext::GetDisplaySize (src/render_graph/compute_execution_context.cpp:8-10). */
int vhr_get_display_size(vhr_context *ctx, uint32_t *width, uint32_t *height);
/* Number of CUDA kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t vhr_kernel_launch_count(vhr_context *ctx);

/* ---- ResourceManager ------------------------------------------------------------------------------------------- */

/* ResourceManager::UpdateGeometry + UpdateBLAS + UpdateTLAS (src/rendering_backend/resource_manager.cpp:291-360,
 * 593-801): uploads the flat Vertex[] (56 B), uint32 indices[] and Primitive[] (120 B) arrays
 * (src/rendering_backend/glsl_common.h:74-99) and builds the acceleration structure on the GPU — an LBVH (Morton
 * codes, radix sort, Karras hierarchy, SAH refit) collapsed into 8-wide quantised nodes — in place of
 * vkCmdBuildAccelerationStructuresKHR. One world-space, opaque, two-sided triangle soup; geometry index = index
 * into `primitives`. Host pointers; returns after the build has been enqueued. */
int vhr_update_geometry(vhr_context *ctx, const void *vertices, uint32_t n_vertices, const uint32_t *indices,
                        uint32_t n_indices, const void *primitives, uint32_t n_primitives);

/* ResourceManager::UploadTextureFromData + GetSampler (resource_manager.cpp:152-193, 821-849, 880-910): uploads one
 * material texture — tightly packed R8G8B8A8 rows, host memory — into the first free slot of textures[2048]
 * (descriptor set 0 binding 4, glsl_common.h:104) and returns that slot (>= 0), the index Material::base_color_texture /
 * metallic_roughness_texture / normal_map name (glsl_common.h:82-91). `sampler_info` = the glTF sampler mapped by the scene
 * loader (scene_loader.cpp:9-38,296-301; values are VkFilter / VkSamplerAddressMode); NULL = the default sampler
 * (LINEAR, REPEAT; resource_manager.cpp:58-69). Border colour is opaque black, one mip level; the ray-traced stages
 * sample LOD 0 (mag filter), anisotropy has no effect without derivatives. VK_FORMAT_R8G8B8A8_SRGB texels are decoded
 * to linear before filtering. Upload textures BEFORE vhr_update_geometry (like the loader does): geometry whose
 * materials name a missing texture is rejected. */
typedef struct vhr_sampler_info {
    int32_t mag_filter, min_filter;            /* VHR_FILTER_* */
    int32_t address_mode_u, address_mode_v;    /* VHR_ADDRESS_MODE_* */
} vhr_sampler_info;
enum { VHR_FILTER_NEAREST = 0, VHR_FILTER_LINEAR = 1 };
enum { VHR_ADDRESS_MODE_REPEAT = 0, VHR_ADDRESS_MODE_MIRRORED_REPEAT = 1, VHR_ADDRESS_MODE_CLAMP_TO_EDGE = 2, VHR_ADDRESS_MODE_CLAMP_TO_BORDER = 3 };
int vhr_upload_texture_from_data(vhr_context *ctx, uint32_t width, uint32_t height, const uint8_t *data, int vk_format,
                                 const vhr_sampler_info *sampler_info);
/* ResourceManager::DestroyResources, texture part (resource_manager.cpp:79-84): frees every texture slot. */
int vhr_destroy_textures(vhr_context *ctx);

/* ResourceManager::UpdatePerFrameUBO (resource_manager.cpp:362-364): `per_frame_data` is the 584-byte PerFrameData
 * of glsl_common.h:59-72. Copied by value; used by every later dispatch until the next call. */
int vhr_update_per_frame_ubo(vhr_context *ctx, const void *per_frame_data, size_t size);

/* ResourceManager::UploadNewStorageImage (resource_manager.cpp:230-263,866-878): returns the first free slot of
 * storage_images[2048] (>= 0) or a negative status. Contents are zero-initialised (documented deviation: the
 * reference leaves them undefined). */
int vhr_upload_new_storage_image(vhr_context *ctx, uint32_t width, uint32_t height, int vk_format);
/* ResourceManager::DestroyStorageImage (resource_manager.cpp:265-269). */
int vhr_destroy_storage_image(vhr_context *ctx, int slot);

/* ---- RenderGraph transient images ------------------------------------------------------------------------------ */

/* RenderGraph::ActualizeResource (src/render_graph/render_graph.cpp:921-977): creates the named image on first
 * mention; width = height = 0 means swapchain-sized. Re-declaring an existing name with another size/format fails
 * (RenderGraph::SanityCheck, render_graph.cpp:980-1021). */
int vhr_actualize_image(vhr_context *ctx, const char *name, uint32_t width, uint32_t height, int vk_format);
/* RenderGraph::DestroyResources (render_graph.cpp:16-68): frees every transient image and the pass/kernel registry. */
int vhr_destroy_transient_resources(vhr_context *ctx);

/* Host <-> device copies of whole images (dense rows). These are the harness' stand-in for the passes outside the
 * hot path (the rasterised G-buffer producer and the composition consumer); `bytes` must equal w*h*texel size.
 * Pinned host memory makes them asynchronous on the context's stream. */
int vhr_image_upload(vhr_context *ctx, const char *name, const void *host, size_t bytes);
int vhr_image_download(vhr_context *ctx, const char *name, void *host, size_t bytes);
int vhr_storage_image_upload(vhr_context *ctx, int slot, const void *host, size_t bytes);
int vhr_storage_image_download(vhr_context *ctx, int slot, void *host, size_t bytes);
/* Transfer queues: the same copies on dedicated upload / download streams, overlapping the passes on the compute
 * stream (the reference keeps up to three frames in flight behind fences, src/rendering_backend/renderer.cpp:103-108,157).
 *   upload_async    starts after every pass enqueued so far (the image's last readers); the first later call that
 *                   binds / blits / copies the image makes the compute stream wait for the upload.
 *   download_async  snapshots the image on the compute stream (device-to-device) and reads the snapshot back on the
 *                   download stream, so later passes may overwrite the image immediately; `*ticket` identifies the
 *                   read-back for vhr_wait_download (reference: vkWaitForFences on the frame's fence). A ticket older
 *                   than the 64 most recent ones counts as complete.
 * Host memory must be pinned for the copies to overlap. vhr_context_synchronize also drains both queues. */
int vhr_image_upload_async(vhr_context *ctx, const char *name, const void *host, size_t bytes);
int vhr_image_download_async(vhr_context *ctx, const char *name, void *host, size_t bytes, uint32_t *ticket);
int vhr_wait_download(vhr_context *ctx, uint32_t ticket);
/* Rows [y0, y1) only (`host_rows` points at row y0): what a rank of the row-band partition moves — its band of the G-buffer up, its band
 * of the result down. The upload follows the rules of vhr_image_upload_async. The download reads the image itself (no device-side
 * snapshot): the compute queue is made to wait for it before anything enqueued later runs. */
int vhr_image_upload_rows_async(vhr_context *ctx, const char *name, const void *host_rows, uint32_t y0, uint32_t y1);
int vhr_image_download_rows_async(vhr_context *ctx, const char *name, void *host_rows, uint32_t y0, uint32_t y1, uint32_t *ticket);
/* `n_blocks` blocks of `block_rows` rows, one every `stride_rows` rows from `first_row`, out of a FULL host image (same row pitch): the rows a
 * rank of the fused partition ray-traces (8-row blocks dealt round-robin) in one strided DMA. */
int vhr_image_upload_blocks_async(vhr_context *ctx, const char *name, const void *host_image, uint32_t first_row, uint32_t block_rows,
                                  uint32_t stride_rows, uint32_t n_blocks);
/* Device pointer of a named image (zero-copy interop, e.g. NCCL halo exchange); NULL if unknown. */
void *vhr_image_device_ptr(vhr_context *ctx, const char *name, uint32_t *width, uint32_t *height, int *vk_format);
void *vhr_storage_image_device_ptr(vhr_context *ctx, int slot, uint32_t *width, uint32_t *height, int *vk_format);

/* ---- pass execution (RenderGraph::Execute*, execution contexts) ------------------------------------------------- */

/* Binds descriptor set 3 of the pass about to execute: the pass' dependencies followed by its outputs, indexed by
 * their `binding` (render_graph.cpp:603-664 CreateComputePass, :893-907/:914-919 vkCmdBindDescriptorSets). */
int vhr_bind_pass_images(vhr_context *ctx, const char *const *names_by_binding, uint32_t count);

/* ComputeExecutionContext::Dispatch (src/render_graph/compute_execution_context.cpp:12-29, .h:20-27). Kernels are
 * looked up by the reference's shader path: "hybrid_render_path/svgf.comp", ".../svgf_atrous_filter.comp",
 * ".../ssao.comp", ".../ssao_blur.comp", ".../ssr.comp". Group size is the shaders' 8x8 (svgf.comp:6): the launcher covers
 * x_groups*8 by y_groups*8 pixels clipped to the image. `push_constants` is SVGFPushConstants (24 B,
 * glsl_common.h:31-39) for the two SVGF kernels, SSAOPushConstants (4 B, :48-50) or NULL (radius 0.75) for SSAO and
 * SSRPushConstants (16 B, :41-46; bound images 0 albedo, 1 normals, 2 motion/metallic-roughness, 3 depth, 4 output) for SSR;
 * a size that does not match fails like the reference's assert (compute_execution_context.h:23).
 * The ssao.comp and ssr.comp dispatches first rewrite a scratch image of the library (16 bytes per texel of the depth image, one per
 * queue, allocated on first use): the 2 x 2 bilinear footprint of every depth texel, which their depth taps read with one load.
 * A svgf_atrous_filter.comp dispatch is deferred: the kernel is launched, on the stream it was recorded for, when anything reads its
 * output (a binding, the next SVGF dispatch, a blit source, a download, vhr_*_device_ptr), writes one of its images in place, frees
 * an input, or calls vhr_context_synchronize, vhr_select_queue or vhr_set_partition; it is never launched if its output is overwritten
 * whole before any read (the reference's last iteration, which the next frame's first iteration overwrites), its output image is
 * destroyed, or the context is destroyed. Every image the caller can observe holds what the immediate launch would have left, and
 * vhr_kernel_launch_count counts the kernel when it is launched. A device pointer exported before the dispatch shows its output only
 * after one of the calls above has launched it. A timestamp (vhr_write_timestamp) written after such a dispatch can
 * come before its kernel. Launches are immediate while a partition is installed, with VHR_OPT_SVGF_FUSED, and once queue 1 exists. */
int vhr_dispatch(vhr_context *ctx, const char *shader_path, uint32_t x_groups, uint32_t y_groups, uint32_t z_groups,
                 const void *push_constants, size_t push_constants_size);

/* RaytracingExecutionContext::TraceRays (src/render_graph/raytracing_execution_context.cpp:4-13) of the pipeline
 * raygen.rgen + miss.rmiss + reflection_miss.rmiss + reflection_hit.rchit (hybrid_render_path.cpp:111-123).
 * Bound images: 0 normals/object ids, 1 depth, 2 shadow+AO (RG16F), 3 reflections (RGBA16F).
 * "Raytracing Pipeline" is the fully ray-traced render path's (src/render_paths/raytraced_render_path.cpp:12-47: raygen.rgen +
 * closesthit.rchit + miss.rmiss + shadow_miss.rmiss, or the *_test_alpha shaders + shadow_anyhit.rahit with
 * VHR_OPT_RAYTRACED_ALPHA_TEST): primary ray, textured / normal-mapped Lambert shading, one shadow ray. Bound image: 0
 * "RaytracedOutput" (B8G8R8A8_UNORM). */
int vhr_trace_rays(vhr_context *ctx, const char *pipeline_name, uint32_t width, uint32_t height);

/* GraphicsExecutionContext::Draw (src/render_graph/graphics_execution_context.cpp:38-41) inside
 * execute_pipeline(<graphics pipeline>) (render_graph.cpp:722-796). The one graphics pipeline on the hot path's
 * consumer side is "Composition Pipeline" (hybrid_render_path.cpp:333-379): composition.vert + composition.frag drawn
 * as one full-screen triangle, Draw(3, 1, 0, 0). `fragment_shader` selects the kernel ("hybrid_render_path/
 * composition.frag"), `specialization_constants` are the pipeline's (shadow_mode, ambient_occlusion_mode,
 * reflection_mode), common.glsl:12-25. Bound images: the nine sampled inputs by binding (0 albedo, 1 normals/ids,
 * 2 motion/metallic-roughness, 3 depth, 4 shadow map, 5 SSAO, 6 SSR, 7 shadow+AO — denoised RGBA16F or raw RG16F —,
 * 8 reflections) followed by colour attachment 0 (RENDER_OUTPUT) at index 9. The attachment may be B8G8R8A8_SRGB (the
 * reference's swapchain: sRGB-encoded on store), B8G8R8A8_UNORM, or R16G16B16A16_SFLOAT (linear HDR radiance, for
 * parity measurements). "raytraced_render_path/composition.frag" (raytraced_render_path.cpp:49-76; no constants) copies
 * bound image 0 (RaytracedOutput) to the attachment at index 1, sRGB-encoding when it is B8G8R8A8_SRGB.
 * Any other shader or draw shape fails with VHR_ERR_INVALID (there is no rasteriser).
 * Both draws write rows [VHR_OPT_ROW_BEGIN, VHR_OPT_ROW_END) of the attachment, under a partition the rank's band. Gathered output:
 * under a partition with world > 1 and VHR_OPT_OUTPUT_RANK = p >= 0, rank p's attachment holds the WHOLE frame after the draw,
 * bit-identical to the single-GPU draw: every other rank stores each texel of its band a second time, with the same bits, into the
 * same texel of rank p's attachment (NVLink peer stores, 4 or 8 B per texel), so the attachment needs rank p's image attached on
 * every rank but p (vhr_image_attach_peer[_pointer]). Every other rank's attachment holds its band as without the option; its rows
 * outside the band are untouched. The call enqueues: a wait for a row read-back of the attachment still in flight, a wait for all
 * ranks (rank p may still be reading its previous frame's output), the one kernel, and a wait for all ranks (every band has landed
 * before anything on rank p reads the attachment). p >= world fails with VHR_ERR_INVALID on every rank; a rank other than p without
 * rank p's attachment fails with VHR_ERR_STATE naming the image and the rank. Both checks run before any flag word is written or
 * waited on. Which path runs is decided on each rank alone, so every rank must set the same output rank and attach p's output the
 * same way: a rank that fails, or that does not gather, leaves the others waiting for flag words it never writes. As with every
 * partitioned call, every rank must issue the same call sequence. */
int vhr_draw(vhr_context *ctx, const char *fragment_shader, const int32_t *specialization_constants, uint32_t n_constants,
             uint32_t vertex_count, uint32_t instance_count, uint32_t first_vertex, uint32_t first_instance);

/* ComputeExecutionContext::Blit* (compute_execution_context.cpp:31-211): same-size, same-format image copies. */
int vhr_blit_storage_to_transient(vhr_context *ctx, int src_slot, const char *dst_name);
int vhr_blit_transient_to_storage(vhr_context *ctx, const char *src_name, int dst_slot);
int vhr_blit_storage_to_storage(vhr_context *ctx, int src_slot, int dst_slot);

/* Per-pass GPU timestamps (render_graph.cpp:143-148 vkCreateQueryPool, :167-182 vkCmdWriteTimestamp, :189-201
 * vkGetQueryPoolResults): a pool of `count` CUDA events recorded on the context's stream. */
int vhr_create_query_pool(vhr_context *ctx, uint32_t count);
/* vkCmdBeginDebugUtilsLabelEXT / vkCmdEndDebugUtilsLabelEXT around every pass node (render_graph.cpp:160-164, :184): an NVTX range named
 * after the pass ("Raytrace Pass", "SVGF Denoise Pass", ...). The kernel-launching calls open their own nested ranges named after the
 * shader path / pipeline name they were given. */
int vhr_cmd_begin_debug_label(vhr_context *ctx, const char *label);
int vhr_cmd_end_debug_label(vhr_context *ctx);
int vhr_write_timestamp(vhr_context *ctx, uint32_t query);
/* Blocks until query `last` has been reached, then writes the elapsed milliseconds between `first` and `last`. */
int vhr_get_query_elapsed_ms(vhr_context *ctx, uint32_t first, uint32_t last, double *out_ms);

/* ---- two queues inside one context: frames in flight ------------------------------------------------------------
 * The reference keeps three frames in flight on one queue (renderer.cpp:103-108, 157) and the driver may run the next frame's
 * first passes under the previous frame's last ones wherever no barrier forbids it. Here that freedom is explicit: queue 0 is
 * the stream the context was created on, queue 1 a second in-order stream the context creates on first use. Every pass, blit,
 * copy and timestamp recorded after vhr_select_queue(q) goes to queue q; the two queues are ordered against each other only by
 * semaphores, like vkQueueSubmit's wait / signal semaphores:
 *   vhr_queue_signal(s)  semaphore s is signalled when everything recorded so far on the selected queue has finished;
 *   vhr_queue_wait(s)    work recorded afterwards on the selected queue starts only after the LAST signal of s recorded so far
 *                        (no-op when s was never signalled).
 * The caller owns the hazards (the Raytrace Pass of frame k+1 may run under the SVGF pass of frame k when it stores into a second
 * set of output images: HybridRenderPath::FrameOverlapped in the host mirrors). Not available while a partition is set. */
#define VHR_MAX_SEMAPHORES 16
int vhr_select_queue(vhr_context *ctx, int queue);          /* 0 or 1 */
int vhr_queue_signal(vhr_context *ctx, int semaphore);
int vhr_queue_wait(vhr_context *ctx, int semaphore);

/* ---- one frame over several GPUs (no counterpart in the reference; SURVEY 8e) ------------------------------------
 * One process per GPU, scene + BVH replicated, every image full-size on every rank. The frame is split by rows:
 *   - SVGF / SSAO / composition work on contiguous row bands: rank r owns rows [band_begin[r], band_begin[r+1]);
 *   - the ray pass deals blocks of `ray_block_rows` rows round-robin over the ranks (traversal cost varies strongly
 *     over the screen, contiguous bands are badly balanced) and every thread stores its result straight into the
 *     OWNER's image over NVLink — compute and the all-to-all that would follow it are one kernel;
 *   - the temporal and a-trous kernels store the boundary rows of their output a second time into the neighbours' copy
 *     of the image (the halo the next kernel there reads): compute and halo exchange are one kernel.
 * Ordering between GPUs is stream-ordered: after such a kernel the library writes a sequence number into the other
 * ranks' flag words (cuStreamWriteValue32 on peer memory) and makes its own stream wait for theirs
 * (cuStreamWaitValue32). No host synchronisation, no NCCL call, no extra copy kernel in the frame. The host keeps
 * issuing the reference's call sequence (vhr_trace_rays, vhr_dispatch, vhr_blit_*) unchanged on every rank.
 * Set-up, once: every rank exports its images (vhr_*_export_ipc), the handles travel between the processes by any
 * means (torch.distributed all_gather_object in multi_gpu.py), every rank attaches the others' (vhr_*_attach_peer),
 * then vhr_set_partition. Requires every band to be at least 64 rows (halos never skip a rank). */
typedef struct vhr_partition {
    uint32_t world, rank;
    uint32_t band_begin[VHR_MAX_RANKS + 1]; /* rows; band_begin[0] = 0, band_begin[world] = image height */
    uint32_t ray_block_rows;                /* 8 = interleaved ray pass (the kernel's tile height); 0 = each rank traces its own band */
    uint32_t motion_halo;                   /* rows of history / moments / previous normals the temporal pass may reach outside the band */
    uint32_t no_exchange_step;              /* a-trous dispatches with this step do not push halos: 16, the reference never reads that output (Q1) */
} vhr_partition;
int vhr_set_partition(vhr_context *ctx, const vhr_partition *partition);       /* NULL: back to single-GPU behaviour */
/* cudaIpcGetMemHandle of the image's buffer; `twin_handle` (may be NULL) exports the second buffer of the
 * double-buffered moments image (allocated on demand). */
int vhr_image_export_ipc(vhr_context *ctx, const char *name, void *handle);
int vhr_storage_image_export_ipc(vhr_context *ctx, int slot, void *handle, void *twin_handle);
int vhr_image_attach_peer(vhr_context *ctx, const char *name, uint32_t rank, const void *handle);
int vhr_storage_image_attach_peer(vhr_context *ctx, int slot, uint32_t rank, const void *handle, const void *twin_handle);
/* The context's flag words (allocated on first use) for the stream-ordered synchronisation. */
int vhr_sync_export_ipc(vhr_context *ctx, void *handle);
int vhr_sync_attach_peer(vhr_context *ctx, uint32_t rank, const void *handle);
/* The same attachments by plain device pointer, for ranks that live in ONE process (several contexts driven by one host
 * thread, on one or several GPUs with peer access enabled): `twin` / flag pointers come from the two getters below. */
int vhr_image_attach_peer_pointer(vhr_context *ctx, const char *name, uint32_t rank, void *device_ptr);
int vhr_storage_image_attach_peer_pointer(vhr_context *ctx, int slot, uint32_t rank, void *device_ptr, void *twin_device_ptr);
int vhr_sync_attach_peer_pointer(vhr_context *ctx, uint32_t rank, void *flag_words);
void *vhr_storage_image_twin_device_ptr(vhr_context *ctx, int slot);     /* second buffer of the moments image (allocated on demand) */
void *vhr_sync_device_ptr(vhr_context *ctx);

/* ---- options that have no counterpart in the reference (documented in DESIGN.md) -------------------------------- */

typedef enum vhr_option {
    VHR_OPT_AO_SPP = 1,            /* AO rays per pixel; reference is hard-wired to 2 (raygen.rgen:45,55) */
    VHR_OPT_TRACE_SHADOWS = 2,     /* 1 (reference) / 0: skip the shadow ray, write 1.0 */
    VHR_OPT_TRACE_AO = 3,          /* 1 (reference) / 0 */
    VHR_OPT_TRACE_REFLECTIONS = 4, /* 1 (reference) / 0: skip the closest-hit ray, write 0 */
    VHR_OPT_ROW_BEGIN = 5,         /* row band [begin, end) this context renders (multi-GPU split); default 0 */
    VHR_OPT_ROW_END = 6,           /* default = image height */
    VHR_OPT_SVGF_FUSED = 7,        /* 1: Dispatch("hybrid_render_path/svgf.comp") runs ONE kernel that does the temporal pass and a-trous
                                      iteration 0 (the tile's integrated[0] texels are computed into shared memory instead of being read
                                      back); the Dispatch("...svgf_atrous_filter.comp") with atrous_step 1 on the same slots that follows
                                      it in the reference's sequence (hybrid_render_path.cpp:299-307) then returns without a launch. The
                                      call sequence and every image are unchanged. Falls back to the two kernels for banded / partitioned
                                      dispatches. Default 0 */
    VHR_OPT_ATROUS_VARIANT = 8,    /* 0: direct-load kernel (the reference's dataflow); 1: tiled kernel; 2 (default): pixel-pair
                                      packed fp32x2 kernel with register-level tap reuse; 3: variant 2's arithmetic in a persistent
                                      CTA with TMA-staged tiles (measured 4-8 % slower than 2 on B200: kept for study) */
    VHR_OPT_DEBUG_REFLECTION_T = 9,/* 1: the ray pass also records the reflection ray's closest-hit distance */
    VHR_OPT_RAYGEN_VARIANT = 10,   /* 0 (default): one thread per pixel, ray kinds in lock step, built for 8 resident blocks / SM (64 registers);
                                      1: persistent warps pulling pixels from a queue, every lane running its pixel's rays back to back;
                                      2 / 3: variant 0 with ptxas' own register choice (72) / without a register cap (117);
                                      4: variant 0 with postponed leaves (the warp runs the triangle block together);
                                      6 / 7: variant 0 launched as one-warp / two-warp CTAs (32 / 16 resident per SM);
                                      8: variant 0 with the CTA's AO rays counting-sorted by direction before they are traced;
                                      9: two-phase kernel — the shadow + AO rays of a 16 x 8 pixel block are generated into shared memory, then traversed with
                                         RAY-level lane refill from that queue (ao_spp 1, 2 or 4; reflections through variant 0 afterwards);
                                      10 / 11: variant 0 built for 10 / 12 resident blocks per SM (48 / 40 registers); 12: 4-byte traversal-stack entries;
                                      13: the shadow ray and the AO rays through one inlined copy of the any-hit traversal;
                                      14 / 15: the first 8 / 12 traversal-stack entries of a thread in shared memory.
                                      Same images in every variant; all measured equal to or slower than 0 on B200, kept for study (DESIGN.md) */
    VHR_OPT_RAYTRACED_ALPHA_TEST = 11,/* the fully ray-traced path's use_anyhit_shader (raytraced_render_path.h:14): 1 selects the pipeline
                                      raygen_test_alpha.rgen + closesthit_test_alpha.rchit + shadow_anyhit.rahit */
    VHR_OPT_BLIT_ALIAS = 12,       /* 1: the three vhr_blit_* calls stop copying. After a blit source and destination show one buffer;
                                      whichever of the two is written next (a kernel output, an upload, another blit) takes the
                                      allocation the destination gave up, so every image always holds what the copy would have left
                                      (copy-on-write). Removes the three copies of the SVGF pass (hybrid_render_path.cpp:309-325: 48 B/px).
                                      Device pointers obtained through vhr_*_device_ptr are invalidated by blits and writes while it is on;
                                      ignored (real copies) while a multi-GPU partition is installed. Default 0 */
    VHR_OPT_OUTPUT_RANK = 13       /* -1 (default): off. p in [0, VHR_MAX_RANKS): under a partition with world > 1 the composition draws
                                      (vhr_draw) gather the whole frame into rank p's render output; see vhr_draw. Every rank must set
                                      the same value and attach p's render output the same way. Ignored without a partition or with
                                      world == 1. Other values: VHR_ERR_INVALID */
} vhr_option;
int vhr_set_option(vhr_context *ctx, int option, int64_t value);
int64_t vhr_get_option(vhr_context *ctx, int option);

/* Extra outputs of the acceleration-structure build and of the ray pass for tests and profiling. */
typedef struct vhr_bvh_stats {
    uint32_t n_triangles;
    uint32_t n_bvh2_nodes;
    uint32_t n_wide_nodes;
    uint32_t max_leaf_size;
    float sah_cost;              /* SAH cost of the wide tree (node cost 1, triangle cost 1) */
    float scene_min[3];
    float scene_max[3];
    float build_ms;              /* device time of the last build */
    uint32_t wide_depth;         /* levels of the wide tree (bounds the traversal stack) */
    uint32_t n_used_slots;       /* child slots in use over all wide nodes (internal children + leaves): n_used_slots / (8 n_wide_nodes) is the
                                    fill rate — every slot of a visited node is slab-tested whether it is used or not */
} vhr_bvh_stats;
int vhr_get_bvh_stats(vhr_context *ctx, vhr_bvh_stats *out);

/* Debug/test entry point: traces `n` explicit rays (origin xyz, tmin, dir xyz, tmax = 8 floats each, host memory).
 * any_hit != 0: out_t[i] = 1 if anything is hit in (tmin, tmax) else 0. Otherwise closest hit: out_t[i] = t or -1,
 * out_ids (optional, 2 x uint32 per ray) = (geometry index, primitive id), out_uv (optional, 2 floats per ray). */
int vhr_trace_explicit(vhr_context *ctx, const float *rays, uint32_t n, int any_hit, float *out_t, uint32_t *out_ids,
                       float *out_uv);

/* Downloads the per-pixel closest-hit distance of the reflection ray written by the last vhr_trace_rays when
 * VHR_OPT_DEBUG_REFLECTION_T is set (float32 per pixel of the display size; -1 = miss or sky). The reference never
 * outputs hit distances (its payloads are 0/1 and radiance); this exists for the hit-distance parity check. */
int vhr_debug_download_reflection_t(vhr_context *ctx, float *host, size_t bytes);

/* Test entry point: runs the per-hit shading code of the passes on hits the caller chooses, so that tests can hold it to a reference
 * on identical hits (the traversal, which decides where a ray hits, is not involved). Record i names a hit by geometry index g
 * (the flat primitive index of vhr_update_geometry), primitive id pid (triangle pid of that primitive) and the barycentrics (u, v) of
 * its vertices 1 and 2, as vhr_trace_explicit returns them. The code runs against the context's state: geometry, normal matrices,
 * the textures of vhr_upload_texture_from_data with their samplers, and the per-frame constants. `out` receives
 * VHR_SHADE_OUT_WORDS 32-bit words per record; words a kind does not write are 0.
 *   VHR_SHADE_TEXTURE           texture(textures[g], (u, v)) at LOD 0 with the slot's sampler (pid, x, y unused): RGBA as 4 floats
 *   VHR_SHADE_REFLECTION        the reflection ray's closest-hit shading (reflection_hit.rchit): RGBA radiance as 4 floats, before
 *                               the RGBA16F store of the ray pass
 *   VHR_SHADE_GBUFFER           the G-buffer pass's texel for a primary hit seen through pixel (x, y): the albedo word (BGRA8), the two
 *                               normals / object-id words (RGBA16F), the two motion / metallic-roughness words (RGBA16F), depth (D32)
 *   VHR_SHADE_GBUFFER_ALPHA     the G-buffer pass's any-hit test (gbuf.frag's discards): 1 = the candidate counts, 0 = discarded
 *   VHR_SHADE_RAYTRACED[_ALPHA] the fully ray-traced path's closest-hit shading (the opaque / the alpha-tested pipeline): the output
 *                               word (BGRA8) when the shadow ray is not occluded, the word when it is, the shadow ray's origin (3 floats)
 *   VHR_SHADE_ANYHIT_ALPHA      the alpha-tested pipeline's any-hit test (shadow_anyhit.rahit): 1 = the candidate counts, 0 = ignored
 * Every record is checked before anything runs: g < the number of primitives and pid < its index_count / 3 (a texture slot in use for
 * VHR_SHADE_TEXTURE); an unknown kind, a NULL array or an invalid record is VHR_ERR_INVALID. VHR_ERR_STATE without per-frame constants
 * or, for the kinds that shade a hit, without geometry; VHR_ERR_CUDA on a VHR_DEVICE_NONE context. Synchronous. */
typedef struct vhr_shade_record {
    uint32_t g;       /* geometry index (VHR_SHADE_TEXTURE: texture slot) */
    uint32_t pid;     /* primitive id within the geometry */
    float u, v;       /* barycentrics of vertices 1 and 2 (VHR_SHADE_TEXTURE: texture coordinates s, t) */
    int32_t x, y;     /* pixel (VHR_SHADE_GBUFFER only) */
} vhr_shade_record;
enum {
    VHR_SHADE_TEXTURE = 0,
    VHR_SHADE_REFLECTION = 1,
    VHR_SHADE_GBUFFER = 2,
    VHR_SHADE_GBUFFER_ALPHA = 3,
    VHR_SHADE_RAYTRACED = 4,
    VHR_SHADE_RAYTRACED_ALPHA = 5,
    VHR_SHADE_ANYHIT_ALPHA = 6
};
#define VHR_SHADE_OUT_WORDS 8
int vhr_debug_shade_hits(vhr_context *ctx, int kind, const vhr_shade_record *records, uint32_t n, uint32_t *out);

/* G-buffer producer as a CUDA primary-ray pass (stand-in for the rasterised "G-Buffer Pass",
 * hybrid_render_path.cpp:13-56; encodings of gbuf.frag:33,43,46-58). Bound images: 0 albedo (BGRA8), 1 normals/ids,
 * 2 motion/metallic-roughness, 3 depth.
 * Without a partition it writes rows [VHR_OPT_ROW_BEGIN, VHR_OPT_ROW_END) of the bound images. Under a partition with world > 1
 * every rank ends with the WHOLE G-buffer, bit-identical to the single-GPU pass: the rank traces the 8-row blocks its ray pass
 * traces (ray_block_rows = 8: blocks b with b % world == rank) or its band (ray_block_rows = 0), and stores every texel, sky
 * clears included, into its own four images and into the same texel of every other rank's (NVLink peer stores, 28 B per texel
 * and peer). So every one of the four bound images needs a peer attached for every other rank (vhr_image_attach_peer[_pointer]);
 * otherwise the call fails with VHR_ERR_STATE before anything is enqueued. After the kernel the call waits for all ranks (their
 * rows have landed before any later pass reads them). Before the kernel it waits for all ranks too when the four images overlap
 * those of the previous partitioned G-buffer pass since vhr_set_partition, or there was none: a peer may still be reading them.
 * When the images differ (alternating G-buffer sets) that pass's trailing wait already ordered every rank's earlier work, so
 * nothing is waited for; work that reads the other set after that pass is the caller's to order. As with every partitioned
 * call, every rank must issue the same call sequence. */
int vhr_gbuffer_pass(vhr_context *ctx, uint32_t width, uint32_t height);

/* Shadow-map producer as a CUDA depth rasteriser (stand-in for the rasterised "Shadow Map Pass", hybrid_render_path.cpp:58-99,
 * depth_prepass.vert/.frag). Bound image 0 is the Shadow Map: D32_SFLOAT, any size (4096 x 4096 in the reference's graph).
 * Draws the world-space triangles of the last vhr_update_geometry, two-sided, through directional_light.projview of the
 * per-frame constants; viewport without Y flip (row 0 = NDC y -1), vertices snapped to 1/256 texel, samples at texel centres
 * with a top-left fill rule, depth kept where 0 <= z <= 1 and combined by max (reverse-Z, cleared to 0). DESIGN.md §2 states
 * the exact arithmetic; the result does not depend on the order of the triangles. projview must be finite with a last row
 * of (0, 0, 0, 1) (an orthographic light, as the scene loader builds) or all zero (a scene without a light: the map is only
 * cleared); anything else is VHR_ERR_INVALID. VHR_ERR_STATE without geometry or per-frame constants; VHR_ERR_CUDA on a
 * VHR_DEVICE_NONE context. VHR_OPT_ROW_BEGIN / END do not apply (the map is not display-sized). Runs on the selected queue.
 * Without a partition, with world == 1, or when the bound map has no peer attached for any other rank, every rank renders
 * the whole map (replicated input, like the acceleration structure). Under a partition with world > 1 and the map attached for
 * every other rank (vhr_image_attach_peer[_pointer]) the pass runs partitioned and every rank ends with the WHOLE map,
 * bit-identical to the single-GPU pass: the map's rows are dealt in blocks of 8 (block b to rank b % world; a rank of a tiny
 * map may own none), each rank projects every triangle but rasterises only the samples of its own rows, clears and fills
 * those rows of its map and stores them into the same rows of every other rank's map (NVLink peer stores, 4 B per texel and
 * peer). The call waits for all ranks before it (a peer may still be reading its map) and after the push (every rank's rows
 * have landed before any later pass reads the map). The cleared-map cases (zero projview, no triangles) run the same way.
 * With the map attached for some other ranks but not all, the call fails with VHR_ERR_STATE naming the missing rank; that
 * check and the ones above run before any flag word is written or waited on. Which path runs is decided on each rank alone, so
 * every rank must attach the map the same way: a rank with every peer attached waits for flag words that a rank with none
 * attached never writes. As with every partitioned call, every rank must issue the same call sequence. */
int vhr_shadow_map_pass(vhr_context *ctx);

#ifdef __cplusplus
}
#endif
#endif /* VHR_B200_H */
