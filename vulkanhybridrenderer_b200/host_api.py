"""ctypes binding of the C++ host (vulkanhybridrenderer_b200/libvhr_host.so): RenderGraph + HybridRenderPath mirrors.

`Renderer` is the headless stand-in for the reference's `Renderer` (src/rendering_backend/renderer.cpp): it owns a
ResourceManager (one vhr_context), a RenderGraph and a HybridRenderPath, loads a scene, switches modes (the ImGui radio
buttons of hybrid_render_path.cpp:394-441) and renders frames. Images are read back through the underlying C-ABI context.
"""
import ctypes as C
import os

import numpy as np

from . import capi
from . import types as T

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvhr_host.so")
SYMBOLS = ["vhrh_last_error", "vhrh_renderer_create", "vhrh_renderer_destroy", "vhrh_context", "vhrh_load_scene", "vhrh_set_modes",
           "vhrh_set_gbuffer_producer", "vhrh_set_shadow_map_producer", "vhrh_render", "vhrh_execution_order", "vhrh_pass_time_ms", "vhrh_svgf_push_constants",
           "vhrh_parse_gltf", "vhrh_parsed_scene_destroy", "vhrh_parsed_scene_counts", "vhrh_parsed_scene_copy", "vhrh_parsed_scene_texture",
           "vhrh_load_gltf", "vhrh_decode_png", "vhrh_set_raytraced_path"]

SHADOW_MODE_RAYTRACED, SHADOW_MODE_RASTERIZED, SHADOW_MODE_OFF = 0, 1, 2
AO_MODE_RAYTRACED, AO_MODE_SSAO, AO_MODE_OFF = 0, 1, 2
REFLECTION_MODE_RAYTRACED, REFLECTION_MODE_SSR, REFLECTION_MODE_OFF = 0, 1, 2
DEVICE_NONE = -1

_lib = None


def lib():
    global _lib
    if _lib is None:
        capi.lib()     # libvhr_b200.so first (the host library links against it by rpath=$ORIGIN)
        if not os.path.exists(LIB_PATH):
            raise capi.VhrError(f"{LIB_PATH} is missing: run `python -m vulkanhybridrenderer_b200.build`")
        L = C.CDLL(LIB_PATH)
        vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int
        L.vhrh_last_error.restype = C.c_char_p
        L.vhrh_renderer_create.argtypes = [i32, vp, u32, u32, C.POINTER(vp)]
        L.vhrh_renderer_destroy.argtypes = [vp]
        L.vhrh_renderer_destroy.restype = None
        L.vhrh_context.argtypes = [vp]
        L.vhrh_context.restype = vp
        L.vhrh_load_scene.argtypes = [vp, vp, u32, vp, u32, vp, u32, u32]
        L.vhrh_set_modes.argtypes = [vp, i32, i32, i32, i32, i32]
        L.vhrh_set_gbuffer_producer.argtypes = [vp, i32]
        L.vhrh_set_shadow_map_producer.argtypes = [vp, i32]
        L.vhrh_render.argtypes = [vp, vp, C.c_size_t, i32]
        L.vhrh_execution_order.argtypes = [vp, C.c_char_p, C.c_size_t]
        L.vhrh_execution_order.restype = u32
        L.vhrh_pass_time_ms.argtypes = [vp, C.c_char_p, i32]
        L.vhrh_pass_time_ms.restype = C.c_double
        L.vhrh_svgf_push_constants.argtypes = [vp, vp]
        L.vhrh_parse_gltf.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.vhrh_parsed_scene_destroy.argtypes = [vp]
        L.vhrh_parsed_scene_destroy.restype = None
        L.vhrh_parsed_scene_counts.argtypes = [vp, C.POINTER(u32)]
        L.vhrh_parsed_scene_copy.argtypes = [vp, vp, vp, vp, vp, vp, vp]
        L.vhrh_parsed_scene_texture.argtypes = [vp, u32, C.POINTER(C.c_int32), vp]
        L.vhrh_load_gltf.argtypes = [vp, C.c_char_p]
        L.vhrh_set_raytraced_path.argtypes = [vp, i32]
        L.vhrh_decode_png.argtypes = [vp, C.c_size_t, C.POINTER(u32), vp, C.c_size_t]
        _lib = L
    return _lib


def _check(rc):
    if rc < 0:
        raise capi.VhrError(f"vhr host status {rc}: {lib().vhrh_last_error().decode()}")
    return rc


class _BorrowedContext(capi.Context):
    """capi.Context view of the renderer's vhr_context (not owned: never destroyed from here)."""

    def __init__(self, handle, width, height):
        self._h = C.c_void_p(handle)
        self.width, self.height = width, height

    def close(self):
        self._h = None


class Renderer:
    def __init__(self, width, height, device=0, stream=None):
        self._r = C.c_void_p()
        _check(lib().vhrh_renderer_create(int(device), C.c_void_p(stream) if stream else None, width, height, C.byref(self._r)))
        self.width, self.height = width, height
        self.ctx = _BorrowedContext(lib().vhrh_context(self._r), width, height)

    def close(self):
        if getattr(self, "_r", None):
            lib().vhrh_renderer_destroy(self._r)
            self._r = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def load_scene(self, scene, prims_per_mesh=0):
        v = np.ascontiguousarray(scene.vertices); i = np.ascontiguousarray(scene.indices, np.uint32); p = np.ascontiguousarray(scene.primitives)
        assert v.dtype == T.Vertex and p.dtype == T.Primitive
        _check(lib().vhrh_load_scene(self._r, capi._ptr(v), len(v), capi._ptr(i), len(i), capi._ptr(p), len(p), prims_per_mesh))

    def load_gltf(self, path):
        """SceneLoader::LoadScene (scene_loader.cpp:336-349): glTF file -> textures + UpdateGeometry. Returns the primitive count."""
        return _check(lib().vhrh_load_gltf(self._r, str(path).encode()))

    def set_modes(self, shadow=SHADOW_MODE_RAYTRACED, ao=AO_MODE_OFF, reflection=REFLECTION_MODE_OFF, denoise=False, svgf_fused=False):
        _check(lib().vhrh_set_modes(self._r, shadow, ao, reflection, int(denoise), int(svgf_fused)))

    def set_raytraced_path(self, use_anyhit_shader=False):
        """Makes the fully ray-traced render path the active one (raytraced_render_path.cpp:11-78)."""
        _check(lib().vhrh_set_raytraced_path(self._r, int(bool(use_anyhit_shader))))

    def set_gbuffer_producer(self, cuda_primary_rays):
        _check(lib().vhrh_set_gbuffer_producer(self._r, 1 if cuda_primary_rays else 0))

    def set_shadow_map_producer(self, cuda_rasteriser):
        """True: the "Shadow Map Pass" node runs the CUDA depth rasteriser (vhr_shadow_map_pass); False: an external producer."""
        _check(lib().vhrh_set_shadow_map_producer(self._r, 1 if cuda_rasteriser else 0))

    def render(self, pfd, gather_statistics=False):
        pfd = np.ascontiguousarray(pfd)
        _check(lib().vhrh_render(self._r, capi._ptr(pfd), pfd.nbytes, int(gather_statistics)))

    def execution_order(self):
        buf = C.create_string_buffer(4096)
        n = lib().vhrh_execution_order(self._r, buf, len(buf))
        return buf.value.decode().split("\n") if n else []

    def pass_time_ms(self, name, last=True):
        return lib().vhrh_pass_time_ms(self._r, name.encode(), int(last))

    def svgf_push_constants(self):
        pc = np.zeros((), T.SVGFPushConstants)
        _check(lib().vhrh_svgf_push_constants(self._r, capi._ptr(pc)))
        return pc


# Camera of vulkan_common.h:33-41 (column-major matrices)
CameraPOD = np.dtype([("perspective", np.float32, (4, 4)), ("transform", np.float32, (4, 4)), ("view", np.float32, (4, 4)),
                      ("yaw", np.float32), ("pitch", np.float32), ("roll", np.float32)])


def parse_gltf(path):
    """SceneLoader::ParseScene through the C++ host: a glTF 2.0 file -> the flat arrays UpdateGeometry consumes. No GPU needed.
    Returns dict(vertices, indices, primitives, prims_per_mesh, camera, light, textures=[(rgba, format, sampler)])."""
    from . import scenes
    h = C.c_void_p()
    _check(lib().vhrh_parse_gltf(str(path).encode(), C.byref(h)))
    try:
        counts = (C.c_uint32 * 5)()
        _check(lib().vhrh_parsed_scene_counts(h, counts))
        nv, ni, npr, nt, nm = (int(c) for c in counts)
        v = np.zeros(nv, T.Vertex); i = np.zeros(ni, np.uint32); p = np.zeros(npr, T.Primitive); ppm = np.zeros(nm, np.uint32)
        cam = np.zeros((), CameraPOD); light = np.zeros((), T.DirectionalLight)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        _check(lib().vhrh_parsed_scene_copy(h, ptr(v), ptr(i), ptr(p), ptr(ppm), ptr(cam), ptr(light)))
        textures = []
        for k in range(nt):
            info = (C.c_int32 * 7)()
            _check(lib().vhrh_parsed_scene_texture(h, k, info, None))
            rgba = np.zeros((info[1], info[0], 4), np.uint8)
            _check(lib().vhrh_parsed_scene_texture(h, k, info, ptr(rgba)))
            textures.append(scenes.Texture(rgba, int(info[2]), tuple(int(x) for x in info[3:7])))
        return dict(vertices=v, indices=i, primitives=p, prims_per_mesh=ppm, camera=cam, light=light, textures=textures)
    finally:
        lib().vhrh_parsed_scene_destroy(h)


def has_stb_image():
    """True when libvhr_host.so was built against the reference's vendored stb_image.h (JPEG and the other stb formats load)."""
    L = lib()
    L.vhrh_has_stb_image.restype = C.c_int
    return bool(L.vhrh_has_stb_image())


def has_cgltf():
    """True when libvhr_host.so was built against the reference's vendored cgltf.h: parse_gltf then parses with it (VHR_GLTF_PARSER=own in the
    environment selects the loader's own reader)."""
    L = lib()
    L.vhrh_has_cgltf.restype = C.c_int
    return bool(L.vhrh_has_cgltf())


def decode_png(data):
    """SceneLoader::DecodePNG: bytes -> [H, W, 4] uint8."""
    buf = np.frombuffer(bytes(data), np.uint8)
    wh = (C.c_uint32 * 2)()
    _check(lib().vhrh_decode_png(buf.ctypes.data_as(C.c_void_p), buf.size, wh, None, 0))
    out = np.zeros((wh[1], wh[0], 4), np.uint8)
    _check(lib().vhrh_decode_png(buf.ctypes.data_as(C.c_void_p), buf.size, wh, out.ctypes.data_as(C.c_void_p), out.nbytes))
    return out
