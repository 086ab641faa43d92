"""ctypes binding of the C-ABI (include/vhr_b200.h -> vulkanhybridrenderer_b200/libvhr_b200.so).

This is the stub a maintainer of a Python harness would write; INTEGRATION.md shows the C++ one. There is no
fallback: a missing library or a missing sm_100 device raises.
"""
import ctypes as C
import os

import numpy as np

from . import types as T

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VHR_LIB_PATH") or os.path.join(_HERE, "libvhr_b200.so")      # VHR_LIB_PATH: development aid (A/B of two builds)

# every symbol include/vhr_b200.h declares (tests check the library exports exactly these)
SYMBOLS = [
    "vhr_context_create", "vhr_context_destroy", "vhr_last_error", "vhr_context_synchronize", "vhr_get_display_size",
    "vhr_kernel_launch_count", "vhr_update_geometry", "vhr_update_per_frame_ubo", "vhr_upload_new_storage_image",
    "vhr_destroy_storage_image", "vhr_actualize_image", "vhr_destroy_transient_resources", "vhr_image_upload",
    "vhr_image_download", "vhr_storage_image_upload", "vhr_storage_image_download", "vhr_image_device_ptr",
    "vhr_storage_image_device_ptr", "vhr_bind_pass_images", "vhr_dispatch", "vhr_trace_rays",
    "vhr_blit_storage_to_transient", "vhr_blit_transient_to_storage", "vhr_blit_storage_to_storage", "vhr_set_option",
    "vhr_get_option", "vhr_get_bvh_stats", "vhr_trace_explicit", "vhr_gbuffer_pass", "vhr_shadow_map_pass", "vhr_create_query_pool",
    "vhr_write_timestamp", "vhr_get_query_elapsed_ms", "vhr_debug_download_reflection_t", "vhr_debug_shade_hits",
    "vhr_image_upload_async", "vhr_image_download_async", "vhr_wait_download", "vhr_draw",
    "vhr_set_partition", "vhr_image_export_ipc", "vhr_storage_image_export_ipc", "vhr_image_attach_peer",
    "vhr_storage_image_attach_peer", "vhr_sync_export_ipc", "vhr_sync_attach_peer",
    "vhr_image_attach_peer_pointer", "vhr_storage_image_attach_peer_pointer", "vhr_sync_attach_peer_pointer",
    "vhr_storage_image_twin_device_ptr", "vhr_sync_device_ptr",
    "vhr_upload_texture_from_data", "vhr_destroy_textures",
    "vhr_select_queue", "vhr_queue_signal", "vhr_queue_wait",
    "vhr_image_upload_rows_async", "vhr_image_download_rows_async", "vhr_image_upload_blocks_async", "vhr_cmd_begin_debug_label", "vhr_cmd_end_debug_label",
]
MAX_RANKS = 8
MAX_SEMAPHORES = 16
IPC_HANDLE_BYTES = 64


class Partition(C.Structure):
    _fields_ = [("world", C.c_uint32), ("rank", C.c_uint32), ("band_begin", C.c_uint32 * (MAX_RANKS + 1)),
                ("ray_block_rows", C.c_uint32), ("motion_halo", C.c_uint32), ("no_exchange_step", C.c_uint32)]


OPT_AO_SPP, OPT_TRACE_SHADOWS, OPT_TRACE_AO, OPT_TRACE_REFLECTIONS = 1, 2, 3, 4
OPT_ROW_BEGIN, OPT_ROW_END, OPT_SVGF_FUSED, OPT_ATROUS_VARIANT, OPT_DEBUG_REFLECTION_T, OPT_RAYGEN_VARIANT = 5, 6, 7, 8, 9, 10
OPT_RAYTRACED_ALPHA_TEST = 11
OPT_BLIT_ALIAS = 12
OPT_OUTPUT_RANK = 13


class SamplerInfo(C.Structure):
    """SamplerInfo of vulkan_common.h:21-26 (VkFilter / VkSamplerAddressMode values)."""
    _fields_ = [("mag_filter", C.c_int32), ("min_filter", C.c_int32), ("address_mode_u", C.c_int32), ("address_mode_v", C.c_int32)]


FILTER_NEAREST, FILTER_LINEAR = 0, 1
ADDRESS_MODE_REPEAT, ADDRESS_MODE_MIRRORED_REPEAT, ADDRESS_MODE_CLAMP_TO_EDGE, ADDRESS_MODE_CLAMP_TO_BORDER = 0, 1, 2, 3


class BvhStats(C.Structure):
    _fields_ = [("n_triangles", C.c_uint32), ("n_bvh2_nodes", C.c_uint32), ("n_wide_nodes", C.c_uint32),
                ("max_leaf_size", C.c_uint32), ("sah_cost", C.c_float), ("scene_min", C.c_float * 3),
                ("scene_max", C.c_float * 3), ("build_ms", C.c_float), ("wide_depth", C.c_uint32), ("n_used_slots", C.c_uint32)]


class VhrError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VhrError(f"{LIB_PATH} is missing: run `python -m vulkanhybridrenderer_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        vp, u32, i32, sz = C.c_void_p, C.c_uint32, C.c_int, C.c_size_t
        L.vhr_context_create.argtypes = [i32, vp, u32, u32, C.POINTER(vp)]
        L.vhr_context_destroy.argtypes = [vp]
        L.vhr_context_destroy.restype = None
        L.vhr_last_error.restype = C.c_char_p
        L.vhr_context_synchronize.argtypes = [vp]
        L.vhr_get_display_size.argtypes = [vp, C.POINTER(u32), C.POINTER(u32)]
        L.vhr_kernel_launch_count.argtypes = [vp]
        L.vhr_kernel_launch_count.restype = C.c_uint64
        L.vhr_update_geometry.argtypes = [vp, vp, u32, vp, u32, vp, u32]
        L.vhr_update_per_frame_ubo.argtypes = [vp, vp, sz]
        L.vhr_upload_texture_from_data.argtypes = [vp, u32, u32, vp, i32, C.POINTER(SamplerInfo)]
        L.vhr_destroy_textures.argtypes = [vp]
        L.vhr_upload_new_storage_image.argtypes = [vp, u32, u32, i32]
        L.vhr_destroy_storage_image.argtypes = [vp, i32]
        L.vhr_actualize_image.argtypes = [vp, C.c_char_p, u32, u32, i32]
        L.vhr_destroy_transient_resources.argtypes = [vp]
        L.vhr_image_upload.argtypes = [vp, C.c_char_p, vp, sz]
        L.vhr_image_download.argtypes = [vp, C.c_char_p, vp, sz]
        L.vhr_image_upload_async.argtypes = [vp, C.c_char_p, vp, sz]
        L.vhr_image_download_async.argtypes = [vp, C.c_char_p, vp, sz, C.POINTER(u32)]
        L.vhr_wait_download.argtypes = [vp, u32]
        L.vhr_image_upload_rows_async.argtypes = [vp, C.c_char_p, vp, u32, u32]
        L.vhr_image_download_rows_async.argtypes = [vp, C.c_char_p, vp, u32, u32, C.POINTER(u32)]
        L.vhr_image_upload_blocks_async.argtypes = [vp, C.c_char_p, vp, u32, u32, u32, u32]
        L.vhr_cmd_begin_debug_label.argtypes = [vp, C.c_char_p]
        L.vhr_cmd_end_debug_label.argtypes = [vp]
        L.vhr_storage_image_upload.argtypes = [vp, i32, vp, sz]
        L.vhr_storage_image_download.argtypes = [vp, i32, vp, sz]
        L.vhr_image_device_ptr.argtypes = [vp, C.c_char_p, C.POINTER(u32), C.POINTER(u32), C.POINTER(i32)]
        L.vhr_image_device_ptr.restype = vp
        L.vhr_storage_image_device_ptr.argtypes = [vp, i32, C.POINTER(u32), C.POINTER(u32), C.POINTER(i32)]
        L.vhr_storage_image_device_ptr.restype = vp
        L.vhr_bind_pass_images.argtypes = [vp, C.POINTER(C.c_char_p), u32]
        L.vhr_dispatch.argtypes = [vp, C.c_char_p, u32, u32, u32, vp, sz]
        L.vhr_trace_rays.argtypes = [vp, C.c_char_p, u32, u32]
        L.vhr_blit_storage_to_transient.argtypes = [vp, i32, C.c_char_p]
        L.vhr_blit_transient_to_storage.argtypes = [vp, C.c_char_p, i32]
        L.vhr_blit_storage_to_storage.argtypes = [vp, i32, i32]
        L.vhr_set_option.argtypes = [vp, i32, C.c_int64]
        L.vhr_get_option.argtypes = [vp, i32]
        L.vhr_get_option.restype = C.c_int64
        L.vhr_get_bvh_stats.argtypes = [vp, C.POINTER(BvhStats)]
        L.vhr_trace_explicit.argtypes = [vp, vp, u32, i32, vp, vp, vp]
        L.vhr_gbuffer_pass.argtypes = [vp, u32, u32]
        L.vhr_shadow_map_pass.argtypes = [vp]
        L.vhr_draw.argtypes = [vp, C.c_char_p, C.POINTER(C.c_int32), u32, u32, u32, u32, u32]
        L.vhr_set_partition.argtypes = [vp, C.POINTER(Partition)]
        L.vhr_image_export_ipc.argtypes = [vp, C.c_char_p, vp]
        L.vhr_storage_image_export_ipc.argtypes = [vp, i32, vp, vp]
        L.vhr_image_attach_peer.argtypes = [vp, C.c_char_p, u32, vp]
        L.vhr_storage_image_attach_peer.argtypes = [vp, i32, u32, vp, vp]
        L.vhr_sync_export_ipc.argtypes = [vp, vp]
        L.vhr_sync_attach_peer.argtypes = [vp, u32, vp]
        L.vhr_image_attach_peer_pointer.argtypes = [vp, C.c_char_p, u32, vp]
        L.vhr_storage_image_attach_peer_pointer.argtypes = [vp, i32, u32, vp, vp]
        L.vhr_sync_attach_peer_pointer.argtypes = [vp, u32, vp]
        L.vhr_storage_image_twin_device_ptr.argtypes = [vp, i32]
        L.vhr_storage_image_twin_device_ptr.restype = vp
        L.vhr_sync_device_ptr.argtypes = [vp]
        L.vhr_sync_device_ptr.restype = vp
        L.vhr_debug_download_reflection_t.argtypes = [vp, vp, sz]
        L.vhr_debug_shade_hits.argtypes = [vp, i32, vp, u32, vp]
        L.vhr_create_query_pool.argtypes = [vp, u32]
        L.vhr_write_timestamp.argtypes = [vp, u32]
        L.vhr_select_queue.argtypes = [vp, i32]
        L.vhr_queue_signal.argtypes = [vp, i32]
        L.vhr_queue_wait.argtypes = [vp, i32]
        L.vhr_get_query_elapsed_ms.argtypes = [vp, u32, u32, C.POINTER(C.c_double)]
        _lib = L
    return _lib


def _check(rc):
    if rc < 0:
        raise VhrError(f"vhr status {rc}: {lib().vhr_last_error().decode()}")
    return rc


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _addr(buf):
    """Host address of a numpy array or a (pinned) torch CPU tensor."""
    if isinstance(buf, np.ndarray):
        return C.c_void_p(buf.ctypes.data), buf.nbytes
    return C.c_void_p(buf.data_ptr()), buf.numel() * buf.element_size()


class Context:
    """Thin object wrapper over vhr_context: one GPU, one stream."""

    def __init__(self, width, height, device=0, stream=None):
        self._h = C.c_void_p()
        _check(lib().vhr_context_create(int(device), C.c_void_p(stream) if stream else None, int(width), int(height), C.byref(self._h)))
        self.width, self.height = int(width), int(height)

    def close(self):
        if getattr(self, "_h", None):
            lib().vhr_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- ResourceManager --
    def update_geometry(self, vertices, indices, primitives):
        v = np.ascontiguousarray(vertices); i = np.ascontiguousarray(indices, np.uint32); p = np.ascontiguousarray(primitives)
        assert v.dtype == T.Vertex and p.dtype == T.Primitive
        _check(lib().vhr_update_geometry(self._h, _ptr(v), len(v), _ptr(i), len(i), _ptr(p), len(p)))

    def upload_texture_from_data(self, rgba8, fmt=T.VK_FORMAT_R8G8B8A8_UNORM, sampler=None):
        """ResourceManager::UploadTextureFromData: [H, W, 4] uint8 -> texture index. sampler = (mag, min, wrap_u, wrap_v) or None."""
        a = np.ascontiguousarray(rgba8, np.uint8)
        assert a.ndim == 3 and a.shape[2] == 4
        si = C.byref(SamplerInfo(*[int(x) for x in sampler])) if sampler is not None else None
        return _check(lib().vhr_upload_texture_from_data(self._h, a.shape[1], a.shape[0], _ptr(a), int(fmt), si))

    def destroy_textures(self):
        _check(lib().vhr_destroy_textures(self._h))

    def load_scene(self, scene):
        """The loader's order (scene_loader.cpp:233-331): textures first, then UpdateGeometry. Texture i of scene.textures
        must land in slot i (materials name slots), which holds on a context without other textures."""
        for i, t in enumerate(getattr(scene, "textures", [])):
            slot = self.upload_texture_from_data(t.rgba, t.format, t.sampler)
            if slot != i:
                raise VhrError(f"texture {i} landed in slot {slot}: destroy_textures() first")
        self.update_geometry(scene.vertices, scene.indices, scene.primitives)

    def update_per_frame_ubo(self, pfd):
        pfd = np.ascontiguousarray(pfd)
        _check(lib().vhr_update_per_frame_ubo(self._h, _ptr(pfd), pfd.nbytes))

    def upload_new_storage_image(self, width, height, fmt):
        return _check(lib().vhr_upload_new_storage_image(self._h, width, height, fmt))

    def destroy_storage_image(self, slot):
        _check(lib().vhr_destroy_storage_image(self._h, slot))

    # -- RenderGraph images --
    def actualize_image(self, name, fmt, width=0, height=0):
        _check(lib().vhr_actualize_image(self._h, name.encode(), width, height, fmt))

    def destroy_transient_resources(self):
        _check(lib().vhr_destroy_transient_resources(self._h))

    def image_upload(self, name, host):
        pageable = isinstance(host, np.ndarray)
        if pageable:
            host = np.ascontiguousarray(host)
        a, n = _addr(host)
        _check(lib().vhr_image_upload(self._h, name.encode(), a, n))
        if pageable:
            self.synchronize()   # pageable source: do not let the caller free it mid-copy

    def image_download_into(self, name, host):
        a, n = _addr(host)
        _check(lib().vhr_image_download(self._h, name.encode(), a, n))

    def image_upload_async(self, name, host):
        """Upload from pinned host memory on the transfer queue; the next pass that binds `name` waits for it."""
        a, n = _addr(host)
        _check(lib().vhr_image_upload_async(self._h, name.encode(), a, n))

    def image_download_async(self, name, host):
        """Read-back on the download queue; returns the ticket for wait_download()."""
        a, n = _addr(host)
        t = C.c_uint32()
        _check(lib().vhr_image_download_async(self._h, name.encode(), a, n, C.byref(t)))
        return t.value

    def image_upload_rows_async(self, name, host_rows, y0, y1):
        """Rows [y0, y1) of `name` from pinned host memory (host_rows starts at row y0) on the transfer queue."""
        a, _ = _addr(host_rows)
        _check(lib().vhr_image_upload_rows_async(self._h, name.encode(), a, int(y0), int(y1)))

    def image_upload_blocks_async(self, name, host_image, first_row, block_rows, stride_rows, n_blocks):
        """Blocks of `block_rows` rows every `stride_rows` rows from `first_row`, out of the FULL pinned host image, in one strided DMA."""
        a, _ = _addr(host_image)
        _check(lib().vhr_image_upload_blocks_async(self._h, name.encode(), a, int(first_row), int(block_rows), int(stride_rows), int(n_blocks)))

    def image_download_rows_async(self, name, host_rows, y0, y1):
        a, _ = _addr(host_rows)
        t = C.c_uint32()
        _check(lib().vhr_image_download_rows_async(self._h, name.encode(), a, int(y0), int(y1), C.byref(t)))
        return t.value

    def debug_label(self, label):
        """Context manager: an NVTX range named after a pass node (vkCmdBegin/EndDebugUtilsLabelEXT, render_graph.cpp:160-164,184)."""
        ctx = self

        class _L:
            def __enter__(self_inner):
                _check(lib().vhr_cmd_begin_debug_label(ctx._h, label.encode()))

            def __exit__(self_inner, *a):
                _check(lib().vhr_cmd_end_debug_label(ctx._h))
        return _L()

    def wait_download(self, ticket):
        _check(lib().vhr_wait_download(self._h, int(ticket)))

    def image_info(self, name):
        w, h, f = C.c_uint32(), C.c_uint32(), C.c_int()
        p = lib().vhr_image_device_ptr(self._h, name.encode(), C.byref(w), C.byref(h), C.byref(f))
        if not p:
            raise VhrError(f"unknown image {name!r}")
        return p, w.value, h.value, f.value

    def storage_image_info(self, slot):
        w, h, f = C.c_uint32(), C.c_uint32(), C.c_int()
        p = lib().vhr_storage_image_device_ptr(self._h, slot, C.byref(w), C.byref(h), C.byref(f))
        if not p:
            raise VhrError(f"unknown storage image {slot}")
        return p, w.value, h.value, f.value

    @staticmethod
    def _host_array(w, h, fmt):
        dt, ch = T.FORMAT_NUMPY[fmt]
        return np.empty((h, w) if ch == 1 else (h, w, ch), dt)

    def image_download(self, name):
        _, w, h, f = self.image_info(name)
        out = self._host_array(w, h, f)
        self.image_download_into(name, out)
        self.synchronize()
        return out

    def storage_image_upload(self, slot, host):
        host = np.ascontiguousarray(host)
        _check(lib().vhr_storage_image_upload(self._h, slot, _ptr(host), host.nbytes))
        self.synchronize()

    def storage_image_download(self, slot):
        _, w, h, f = self.storage_image_info(slot)
        out = self._host_array(w, h, f)
        _check(lib().vhr_storage_image_download(self._h, slot, _ptr(out), out.nbytes))
        self.synchronize()
        return out

    # -- pass execution --
    def bind_pass_images(self, names):
        arr = (C.c_char_p * len(names))(*[n.encode() for n in names])
        _check(lib().vhr_bind_pass_images(self._h, arr, len(names)))

    def dispatch(self, shader, xg, yg, zg=1, push_constants=None):
        if push_constants is None:
            _check(lib().vhr_dispatch(self._h, shader.encode(), xg, yg, zg, None, 0))
        else:
            pc = np.ascontiguousarray(push_constants)
            _check(lib().vhr_dispatch(self._h, shader.encode(), xg, yg, zg, _ptr(pc), pc.nbytes))

    def trace_rays(self, width, height, pipeline="Raytrace Pipeline"):
        _check(lib().vhr_trace_rays(self._h, pipeline.encode(), width, height))

    def draw(self, fragment_shader, specialization_constants, vertex_count=3, instance_count=1, first_vertex=0, first_instance=0):
        """GraphicsExecutionContext::Draw for the composition pipeline (see vhr_draw)."""
        sc = (C.c_int32 * len(specialization_constants))(*[int(v) for v in specialization_constants])
        _check(lib().vhr_draw(self._h, fragment_shader.encode(), sc, len(specialization_constants), vertex_count, instance_count,
                              first_vertex, first_instance))

    # -- one frame over several GPUs (include/vhr_b200.h) --
    def set_partition(self, world, rank, band_begin, ray_block_rows=8, motion_halo=8, no_exchange_step=16):
        p = Partition()
        p.world, p.rank = world, rank
        if len(band_begin) > MAX_RANKS + 1:
            raise VhrError(f"partition over {len(band_begin) - 1} ranks (max {MAX_RANKS})")
        for i, b in enumerate(band_begin):
            p.band_begin[i] = int(b)
        p.ray_block_rows, p.motion_halo, p.no_exchange_step = ray_block_rows, motion_halo, no_exchange_step
        _check(lib().vhr_set_partition(self._h, C.byref(p)))

    def clear_partition(self):
        _check(lib().vhr_set_partition(self._h, None))

    def image_export_ipc(self, name):
        h = C.create_string_buffer(IPC_HANDLE_BYTES)
        _check(lib().vhr_image_export_ipc(self._h, name.encode(), h))
        return h.raw

    def storage_image_export_ipc(self, slot, twin=False):
        h, t = C.create_string_buffer(IPC_HANDLE_BYTES), C.create_string_buffer(IPC_HANDLE_BYTES)
        _check(lib().vhr_storage_image_export_ipc(self._h, int(slot), h, t if twin else None))
        return (h.raw, t.raw) if twin else (h.raw, None)

    def image_attach_peer(self, name, rank, handle):
        _check(lib().vhr_image_attach_peer(self._h, name.encode(), rank, C.create_string_buffer(handle, IPC_HANDLE_BYTES)))

    def storage_image_attach_peer(self, slot, rank, handle, twin_handle=None):
        t = C.create_string_buffer(twin_handle, IPC_HANDLE_BYTES) if twin_handle else None
        _check(lib().vhr_storage_image_attach_peer(self._h, int(slot), rank, C.create_string_buffer(handle, IPC_HANDLE_BYTES), t))

    def sync_export_ipc(self):
        h = C.create_string_buffer(IPC_HANDLE_BYTES)
        _check(lib().vhr_sync_export_ipc(self._h, h))
        return h.raw

    def sync_attach_peer(self, rank, handle):
        _check(lib().vhr_sync_attach_peer(self._h, rank, C.create_string_buffer(handle, IPC_HANDLE_BYTES)))

    def gbuffer_pass(self, width, height):
        _check(lib().vhr_gbuffer_pass(self._h, width, height))

    def shadow_map_pass(self):
        """Rasterises the scene into bound image 0 (the D32 Shadow Map) from directional_light.projview (vhr_shadow_map_pass)."""
        _check(lib().vhr_shadow_map_pass(self._h))

    def blit_storage_to_transient(self, src, dst):
        _check(lib().vhr_blit_storage_to_transient(self._h, src, dst.encode()))

    def blit_transient_to_storage(self, src, dst):
        _check(lib().vhr_blit_transient_to_storage(self._h, src.encode(), dst))

    def blit_storage_to_storage(self, src, dst):
        _check(lib().vhr_blit_storage_to_storage(self._h, src, dst))

    def set_option(self, opt, value):
        _check(lib().vhr_set_option(self._h, opt, int(value)))

    def get_option(self, opt):
        return lib().vhr_get_option(self._h, opt)

    # ---- two queues (frames in flight) --------------------------------------------------------------------------------
    def select_queue(self, queue):
        _check(lib().vhr_select_queue(self._h, int(queue)))

    def queue_signal(self, semaphore):
        _check(lib().vhr_queue_signal(self._h, int(semaphore)))

    def queue_wait(self, semaphore):
        _check(lib().vhr_queue_wait(self._h, int(semaphore)))

    def synchronize(self):
        _check(lib().vhr_context_synchronize(self._h))

    @property
    def kernel_launches(self):
        return lib().vhr_kernel_launch_count(self._h)

    def bvh_stats(self):
        s = BvhStats()
        _check(lib().vhr_get_bvh_stats(self._h, C.byref(s)))
        return s

    def download_reflection_t(self):
        out = np.empty((self.height, self.width), np.float32)
        _check(lib().vhr_debug_download_reflection_t(self._h, _ptr(out), out.nbytes))
        return out

    def trace_explicit(self, rays, any_hit):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        n = len(rays)
        t = np.empty(n, np.float32)
        ids = np.empty((n, 2), np.uint32)
        uv = np.empty((n, 2), np.float32)
        _check(lib().vhr_trace_explicit(self._h, _ptr(rays), n, int(bool(any_hit)), _ptr(t), _ptr(ids), _ptr(uv)))
        return t, ids, uv

    def shade_hits(self, kind, records):
        """vhr_debug_shade_hits: the per-hit shading of `kind` (types.SHADE_*) on the records (array of types.ShadeRecord).
        Returns [n, types.SHADE_OUT_WORDS] uint32: the output words of each record (include/vhr_b200.h)."""
        rec = np.ascontiguousarray(records, T.ShadeRecord).reshape(-1)
        out = np.zeros((len(rec), T.SHADE_OUT_WORDS), np.uint32)
        _check(lib().vhr_debug_shade_hits(self._h, int(kind), _ptr(rec), len(rec), _ptr(out)))
        return out
