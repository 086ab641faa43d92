// peer.cu — one frame over the GPUs of an NVSwitch box: CUDA IPC mapping of the other ranks' images, the row
// partition, and the stream-ordered flag exchange that orders kernels across GPUs (include/vhr_b200.h, "one frame over
// several GPUs"). The data itself moves inside the compute kernels (peer stores in trace_kernels.cu / svgf_kernels.cu).
#include <cuda.h>
#include <string.h>

#include "vhr_internal.h"

namespace vhr {

namespace {
typedef CUresult (*WriteValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
typedef CUresult (*WaitValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
WriteValue32Fn g_write32 = nullptr;
WaitValue32Fn g_wait32 = nullptr;

int load_driver_entry_points() {
    if (g_write32 && g_wait32) return VHR_OK;
    cudaDriverEntryPointQueryResult q;
    void *fn = nullptr;
    VHR_CUDA_CHECK(cudaGetDriverEntryPoint("cuStreamWriteValue32", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) return fail(VHR_ERR_CUDA, "cuStreamWriteValue32 is not available in this driver");
    g_write32 = (WriteValue32Fn)fn;
    fn = nullptr;
    VHR_CUDA_CHECK(cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) return fail(VHR_ERR_CUDA, "cuStreamWaitValue32 is not available in this driver");
    g_wait32 = (WaitValue32Fn)fn;
    return VHR_OK;
}

int ensure_flags(vhr_context *ctx) {
    if (ctx->sync_flags) return VHR_OK;
    VHR_CUDA_CHECK(cudaMalloc(&ctx->sync_flags, 2 * VHR_MAX_RANKS * sizeof(uint32_t)));
    VHR_CUDA_CHECK(cudaMemset(ctx->sync_flags, 0, 2 * VHR_MAX_RANKS * sizeof(uint32_t)));
    return VHR_OK;
}

int open_handle(vhr_context *ctx, const void *handle, void **out) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    VHR_CUDA_CHECK(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->ipc_opened.push_back(*out);
    return VHR_OK;
}
int export_ptr(void *ptr, void *handle) {
    cudaIpcMemHandle_t h;
    VHR_CUDA_CHECK(cudaIpcGetMemHandle(&h, ptr));
    memcpy(handle, &h, sizeof(h));
    return VHR_OK;
}
int signal_and_wait(vhr_context *ctx, uint32_t base, uint32_t seq, const int *ranks, int n) {
    if (int rc = load_driver_entry_points()) return rc;
    const Partition &pt = ctx->part;
    for (int i = 0; i < n; ++i) {
        uint32_t *dst = ctx->peer_flags[ranks[i]];
        if (!dst) return fail(VHR_ERR_STATE, "rank %d's flag words are not attached (vhr_sync_attach_peer)", ranks[i]);
        // default flags: the write is ordered after the preceding kernel's (peer) stores with a system-scope fence
        CUresult r = g_write32((CUstream)ctx->stream, (CUdeviceptr)(dst + base + pt.rank), seq, 0);
        if (r != CUDA_SUCCESS) return fail(VHR_ERR_CUDA, "cuStreamWriteValue32 failed (%d)", (int)r);
    }
    for (int i = 0; i < n; ++i) {
        CUresult r = g_wait32((CUstream)ctx->stream, (CUdeviceptr)(ctx->sync_flags + base + ranks[i]), seq, CU_STREAM_WAIT_VALUE_GEQ);
        if (r != CUDA_SUCCESS) return fail(VHR_ERR_CUDA, "cuStreamWaitValue32 failed (%d)", (int)r);
    }
    return VHR_OK;
}
}  // namespace

int peer_sync_neighbours(vhr_context *ctx) {
    const Partition &pt = ctx->part;
    if (!pt.enabled || pt.world == 1) return VHR_OK;
    int ranks[2], n = 0;
    if (pt.rank > 0) ranks[n++] = pt.rank - 1;
    if (pt.rank + 1 < pt.world) ranks[n++] = pt.rank + 1;
    return signal_and_wait(ctx, VHR_MAX_RANKS, ++ctx->seq_halo, ranks, n);
}

int peer_sync_all(vhr_context *ctx) {
    const Partition &pt = ctx->part;
    if (!pt.enabled || pt.world == 1) return VHR_OK;
    int ranks[VHR_MAX_RANKS], n = 0;
    for (int r = 0; r < pt.world; ++r)
        if (r != pt.rank) ranks[n++] = r;
    return signal_and_wait(ctx, 0, ++ctx->seq_ray, ranks, n);
}

HaloPush halo_push_for(vhr_context *ctx, Image *out, bool twin, int rows) {
    HaloPush hp;
    const Partition &pt = ctx->part;
    if (!pt.enabled || pt.world == 1 || rows <= 0) return hp;
    void **peers = twin ? out->peer_twin : out->peer;
    if (pt.rank > 0) hp.up = peers[pt.rank - 1];
    if (pt.rank + 1 < pt.world) hp.down = peers[pt.rank + 1];
    hp.rows = rows;
    return hp;
}

void peer_close_all(vhr_context *ctx) {
    for (void *p : ctx->ipc_opened) cudaIpcCloseMemHandle(p);
    ctx->ipc_opened.clear();
    if (ctx->sync_flags) cudaFree(ctx->sync_flags);
    ctx->sync_flags = nullptr;
}

}  // namespace vhr

using namespace vhr;

#define VHR_NEED_DEVICE(ctx)                                                                                     \
    do {                                                                                                         \
        if (!(ctx)) return fail(VHR_ERR_INVALID, "ctx is NULL");                                                 \
        if ((ctx)->device < 0) return fail(VHR_ERR_CUDA, "%s: context was created with VHR_DEVICE_NONE (no GPU work possible, no CPU fallback)", __func__); \
        VHR_CUDA_CHECK(cudaSetDevice((ctx)->device));                                                            \
    } while (0)

static Image *transient(vhr_context *ctx, const char *name) {
    if (!name) return nullptr;
    auto it = ctx->transient.find(name);
    return it == ctx->transient.end() ? nullptr : &it->second;
}

extern "C" {

int vhr_set_partition(vhr_context *ctx, const vhr_partition *p) {
    if (!ctx) return fail(VHR_ERR_INVALID, "ctx is NULL");
    for (Image *&im : ctx->gbuffer_peer_written) im = nullptr;      // the next partitioned G-buffer pass starts with a leading sync
    if (!p) {      // back to single-GPU behaviour: the whole image is the dispatch range again
        ctx->part = Partition();
        ctx->opt.row_begin = 0;
        ctx->opt.row_end = -1;
        return VHR_OK;
    }
    if (ctx->stream != ctx->queue[0]) return fail(VHR_ERR_STATE, "partition: select queue 0 first (the peer flag words are ordered on it)");
    if (p->world < 1 || p->world > VHR_MAX_RANKS || p->rank >= p->world) return fail(VHR_ERR_INVALID, "partition: rank %u of %u (max %d ranks)", p->rank, p->world, VHR_MAX_RANKS);
    if (p->band_begin[0] != 0 || p->band_begin[p->world] != ctx->height) return fail(VHR_ERR_INVALID, "partition: bands must cover rows [0, %u)", ctx->height);
    if (p->ray_block_rows != 0 && p->ray_block_rows != 8) return fail(VHR_ERR_INVALID, "partition: ray_block_rows must be 0 or 8 (the ray kernel's tile height)");
    if (p->motion_halo > 64) return fail(VHR_ERR_INVALID, "partition: motion_halo %u > 64 rows", p->motion_halo);
    for (uint32_t r = 0; r < p->world; ++r)
        if (p->world > 1 && p->band_begin[r + 1] < p->band_begin[r] + 64)
            return fail(VHR_ERR_INVALID, "partition: band %u has %d rows; every band must hold at least 64 (halos never skip a rank)", r,
                        (int)p->band_begin[r + 1] - (int)p->band_begin[r]);
    // copy-free blits (VHR_OPT_BLIT_ALIAS) are suspended while a partition is installed — the peers hold mappings of fixed buffers — so every
    // image that still shares a buffer with a blit partner gets its own copy now
    if (ctx->device >= 0) {
        if (int rc = launch_pending_atrous(ctx)) return rc;      // peers will store into these images unseen: no deferred dispatch
        for (auto &kv : ctx->transient)
            if (int rc = make_writable(ctx, &kv.second, false)) return rc;
        for (auto &im : ctx->storage)
            if (im.used)
                if (int rc = make_writable(ctx, &im, false)) return rc;
    }
    Partition pt;
    pt.enabled = true; pt.world = (int)p->world; pt.rank = (int)p->rank;
    for (uint32_t r = 0; r <= p->world; ++r) pt.band_begin[r] = (int)p->band_begin[r];
    pt.ray_block_rows = (int)p->ray_block_rows; pt.motion_halo = (int)p->motion_halo; pt.no_exchange_step = (int)p->no_exchange_step;
    ctx->part = pt;
    // the band doubles as the dispatch range of every banded kernel
    ctx->opt.row_begin = pt.band_begin[pt.rank];
    ctx->opt.row_end = pt.band_begin[pt.rank + 1];
    return VHR_OK;
}

int vhr_image_export_ipc(vhr_context *ctx, const char *name, void *handle) {
    VHR_NEED_DEVICE(ctx);
    Image *im = transient(ctx, name);
    if (!im || !handle) return fail(VHR_ERR_INVALID, "export: unknown image '%s'", name ? name : "(null)");
    if (int rc = make_writable(ctx, im, false)) return rc;        // a buffer shared with a blit partner is not this image's to hand out
    return export_ptr(im->ptr, handle);
}
int vhr_storage_image_export_ipc(vhr_context *ctx, int slot, void *handle, void *twin_handle) {
    VHR_NEED_DEVICE(ctx);
    Image *im = storage_slot(ctx, slot);
    if (!im || !handle) return fail(VHR_ERR_INVALID, "export: storage image %d does not exist", slot);
    if (int rc = make_writable(ctx, im, false)) return rc;
    if (int rc = export_ptr(im->ptr, handle)) return rc;
    if (twin_handle) {
        if (!im->twin) {
            VHR_CUDA_CHECK(cudaMalloc(&im->twin, im->bytes));
            VHR_CUDA_CHECK(cudaMemsetAsync(im->twin, 0, im->bytes, ctx->stream));
        }
        return export_ptr(im->twin, twin_handle);
    }
    return VHR_OK;
}
int vhr_image_attach_peer(vhr_context *ctx, const char *name, uint32_t rank, const void *handle) {
    VHR_NEED_DEVICE(ctx);
    Image *im = transient(ctx, name);
    if (!im || !handle || rank >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "attach: unknown image '%s' or rank %u", name ? name : "(null)", rank);
    return open_handle(ctx, handle, &im->peer[rank]);
}
int vhr_storage_image_attach_peer(vhr_context *ctx, int slot, uint32_t rank, const void *handle, const void *twin_handle) {
    VHR_NEED_DEVICE(ctx);
    Image *im = storage_slot(ctx, slot);
    if (!im || !handle || rank >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "attach: storage image %d does not exist or rank %u", slot, rank);
    if (int rc = open_handle(ctx, handle, &im->peer[rank])) return rc;
    if (twin_handle) return open_handle(ctx, twin_handle, &im->peer_twin[rank]);
    return VHR_OK;
}
int vhr_sync_export_ipc(vhr_context *ctx, void *handle) {
    VHR_NEED_DEVICE(ctx);
    if (!handle) return fail(VHR_ERR_INVALID, "NULL handle");
    if (int rc = ensure_flags(ctx)) return rc;
    return export_ptr(ctx->sync_flags, handle);
}
int vhr_sync_attach_peer(vhr_context *ctx, uint32_t rank, const void *handle) {
    VHR_NEED_DEVICE(ctx);
    if (!handle || rank >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "attach: rank %u", rank);
    if (int rc = ensure_flags(ctx)) return rc;
    void *p = nullptr;
    if (int rc = open_handle(ctx, handle, &p)) return rc;
    ctx->peer_flags[rank] = (uint32_t *)p;
    return VHR_OK;
}

int vhr_image_attach_peer_pointer(vhr_context *ctx, const char *name, uint32_t rank, void *device_ptr) {
    VHR_NEED_DEVICE(ctx);
    Image *im = transient(ctx, name);
    if (!im || !device_ptr || rank >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "attach: unknown image '%s' or rank %u", name ? name : "(null)", rank);
    im->peer[rank] = device_ptr;
    return VHR_OK;
}
int vhr_storage_image_attach_peer_pointer(vhr_context *ctx, int slot, uint32_t rank, void *device_ptr, void *twin_device_ptr) {
    VHR_NEED_DEVICE(ctx);
    Image *im = storage_slot(ctx, slot);
    if (!im || !device_ptr || rank >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "attach: storage image %d does not exist or rank %u", slot, rank);
    im->peer[rank] = device_ptr;
    im->peer_twin[rank] = twin_device_ptr;
    return VHR_OK;
}
int vhr_sync_attach_peer_pointer(vhr_context *ctx, uint32_t rank, void *flag_words) {
    VHR_NEED_DEVICE(ctx);
    if (!flag_words || rank >= VHR_MAX_RANKS) return fail(VHR_ERR_INVALID, "attach: rank %u", rank);
    if (int rc = ensure_flags(ctx)) return rc;
    ctx->peer_flags[rank] = (uint32_t *)flag_words;
    return VHR_OK;
}
void *vhr_storage_image_twin_device_ptr(vhr_context *ctx, int slot) {
    if (!ctx || ctx->device < 0) return nullptr;
    Image *im = storage_slot(ctx, slot);
    if (!im) return nullptr;
    if (!im->twin) {
        if (cudaSetDevice(ctx->device) != cudaSuccess || cudaMalloc(&im->twin, im->bytes) != cudaSuccess) return nullptr;
        cudaMemsetAsync(im->twin, 0, im->bytes, ctx->stream);
    }
    return im->twin;
}
void *vhr_sync_device_ptr(vhr_context *ctx) {
    if (!ctx || ctx->device < 0) return nullptr;
    if (cudaSetDevice(ctx->device) != cudaSuccess || ensure_flags(ctx) != VHR_OK) return nullptr;
    return ctx->sync_flags;
}

}  // extern "C"
