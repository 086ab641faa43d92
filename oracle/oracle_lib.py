"""ctypes binding of the CPU oracle (oracle/_build/libvhr_oracle.so). TEST INFRASTRUCTURE ONLY.

Builds the library with `make -C oracle` when it is missing or stale. Used by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs — never by the product path.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from vulkanhybridrenderer_b200 import types as T

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))  # repo root (this file lives in oracle/)
_ORACLE_DIR = os.path.join(_ROOT, "oracle")
_SO = os.path.join(_ORACLE_DIR, "_build", "libvhr_oracle.so")
_SRCS = ["oracle_common.h", "oracle_svgf.cpp", "oracle_rt.cpp", "oracle_composition.cpp", "oracle_ssr.cpp", "Makefile"]


def build(force=False):
    stale = force or not os.path.exists(_SO)
    if not stale:
        so_m = os.path.getmtime(_SO)
        stale = any(os.path.getmtime(os.path.join(_ORACLE_DIR, s)) > so_m for s in _SRCS)
    if stale:
        env = dict(os.environ)
        env.pop("CXX", None)
        subprocess.run(["make", "-C", _ORACLE_DIR], check=True, env=env, capture_output=True)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _declare(_lib)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _declare(L):
    vp = C.c_void_p
    L.vo_svgf_temporal.argtypes = [vp, C.c_int, C.c_int] + [vp] * 8
    L.vo_svgf_atrous.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.vo_svgf_state_create.restype = vp
    L.vo_svgf_state_create.argtypes = [C.c_int, C.c_int]
    L.vo_svgf_state_destroy.argtypes = [vp]
    L.vo_svgf_state_image.restype = C.POINTER(C.c_uint16)
    L.vo_svgf_state_image.argtypes = [vp, C.c_int]
    L.vo_svgf_pass.argtypes = [vp] * 8
    L.vo_ssao.argtypes = [vp, C.c_int, C.c_int, C.c_float, vp, vp, vp]
    L.vo_ssao_blur.argtypes = [vp, C.c_int, C.c_int, vp, vp]
    L.vo_composition.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp, C.c_int, vp]
    L.vo_ssr.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, vp, vp, vp, vp, vp]
    L.vo_seed_thread.restype = C.c_uint32
    L.vo_seed_thread.argtypes = [C.c_uint32]
    L.vo_random01.restype = C.c_float
    L.vo_random01.argtypes = [C.POINTER(C.c_uint32)]
    L.vo_uniform_sample_cone.argtypes = [C.c_float, C.c_float, C.c_float, vp]
    L.vo_cosine_hemisphere.argtypes = [C.c_float, C.c_float, vp]
    L.vo_onb.argtypes = [vp, vp]
    L.vo_f2h.restype = C.c_uint16
    L.vo_f2h.argtypes = [C.c_float]
    L.vo_h2f.restype = C.c_float
    L.vo_h2f.argtypes = [C.c_uint16]
    L.vo_sizeof.restype = C.c_int
    L.vo_sizeof.argtypes = [C.c_int]
    L.vo_scene_create.restype = vp
    L.vo_scene_create.argtypes = [vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32]
    L.vo_scene_destroy.argtypes = [vp]
    L.vo_scene_add_texture.restype = C.c_int
    L.vo_scene_add_texture.argtypes = [vp, C.c_uint32, C.c_uint32, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.vo_sample_texture.argtypes = [vp, C.c_int, C.c_float, C.c_float, vp]
    L.vo_scene_num_triangles.restype = C.c_uint32
    L.vo_scene_num_triangles.argtypes = [vp]
    L.vo_trace_any.restype = C.c_int
    L.vo_trace_any.argtypes = [vp, vp, vp, C.c_float, C.c_float]
    L.vo_trace_closest.restype = C.c_int
    L.vo_trace_closest.argtypes = [vp, vp, vp, C.c_float, C.c_float, vp, vp]
    L.vo_raygen.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]
    L.vo_raytraced.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp]
    L.vo_raygen_pixel_rays.restype = C.c_int
    L.vo_raygen_pixel_rays.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp]
    L.vo_brute_force.argtypes = [vp, vp, vp, C.c_float, C.c_float, vp]
    L.vo_gbuffer.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]
    L.vo_shade_hits.restype = C.c_int
    L.vo_shade_hits.argtypes = [vp, vp, C.c_int, vp, C.c_uint32, vp]


def set_num_threads(n=0):
    """Sets the OpenMP thread count of the oracle's loops (n <= 0: leave it) and returns the count the runtime will use."""
    L = lib()
    L.vo_set_num_threads.restype = C.c_int
    L.vo_set_num_threads.argtypes = [C.c_int]
    return int(L.vo_set_num_threads(int(n)))


def _h(a):
    """float16 array -> contiguous uint16 view"""
    a = np.ascontiguousarray(a)
    assert a.dtype == np.float16
    return a.view(np.uint16)


def svgf_temporal(pfd, normals, motion, rt, prev_normals, history, moments_in):
    H, W = normals.shape[:2]
    integ = np.empty((H, W, 4), np.float16)
    mom = np.empty((H, W, 2), np.float16)
    lib().vo_svgf_temporal(_p(pfd), W, H, _p(_h(normals)), _p(_h(motion)), _p(_h(rt)), _p(_h(prev_normals)),
                           _p(_h(history)), _p(_h(moments_in)), _p(integ), _p(mom))
    return integ, mom


def svgf_atrous(pfd, normals, integ_in, step):
    H, W = normals.shape[:2]
    out = np.empty((H, W, 4), np.float16)
    lib().vo_svgf_atrous(_p(pfd), W, H, int(step), _p(_h(normals)), _p(_h(integ_in)), _p(out))
    return out


class SvgfState:
    """The five persistent SVGF images + ping-pong bookkeeping of hybrid_render_path.cpp:245-331."""

    def __init__(self, W, H):
        self.W, self.H = W, H
        self._s = lib().vo_svgf_state_create(W, H)

    def __del__(self):
        if getattr(self, "_s", None):
            lib().vo_svgf_state_destroy(self._s)
            self._s = None

    def image(self, which):
        ch = 2 if which == 4 else 4
        ptr = lib().vo_svgf_state_image(self._s, which)
        return np.ctypeslib.as_array(ptr, shape=(self.H, self.W, ch)).view(np.float16)

    def run(self, pfd, normals, motion, rt, want_iters=True):
        W, H = self.W, self.H
        den = np.empty((H, W, 4), np.float16)
        iters = np.empty((5, H, W, 4), np.float16) if want_iters else None
        temporal = np.empty((H, W, 4), np.float16)
        lib().vo_svgf_pass(self._s, _p(pfd), _p(_h(normals)), _p(_h(motion)), _p(_h(rt)), _p(den), _p(iters), _p(temporal))
        return den, iters, temporal


def ssao(pfd, depth, normals, radius=0.75):
    H, W = depth.shape[:2]
    out = np.empty((H, W, 4), np.float16)
    d = np.ascontiguousarray(depth, np.float32)
    lib().vo_ssao(_p(pfd), W, H, float(radius), _p(d), _p(_h(normals)), _p(out))
    return out


def ssao_blur(pfd, raw):
    H, W = raw.shape[:2]
    out = np.empty((H, W, 4), np.float16)
    lib().vo_ssao_blur(_p(pfd), W, H, _p(_h(raw)), _p(out))
    return out


def ssr(pfd, albedo, normals, motion, depth, ray_distance=25.0, step_size=0.1, thickness=0.5, bsearch_steps=10, rows=None):
    """ssr.comp over rows [y0, y1) (default: the whole frame); defaults = hybrid_render_path.cpp:203-208."""
    H, W = depth.shape[:2]
    y0, y1 = (0, H) if rows is None else rows
    out = np.zeros((H, W, 4), np.float16)
    a8 = np.ascontiguousarray(albedo, np.uint8)
    d = np.ascontiguousarray(depth, np.float32)
    lib().vo_ssr(_p(pfd), W, H, y0, y1, float(ray_distance), float(step_size), float(thickness), int(bsearch_steps), _p(a8), _p(_h(normals)),
                 _p(_h(motion)), _p(d), _p(out))
    return out


def composition(pfd, albedo, normals, motion, depth, rt, shadow_mode=0, ao_mode=0, reflection_mode=2, ssao_img=None, ssr_img=None,
                refl=None, shadow_map=None, out_format=T.VK_FORMAT_R16G16B16A16_SFLOAT):
    """composition.frag over a whole frame. `rt` is the raw RG16F or the denoised RGBA16F shadow/AO image (binding 7)."""
    H, W = depth.shape[:2]
    zero4 = np.zeros((H, W, 4), np.float16)
    ssao_img = zero4 if ssao_img is None else _h(ssao_img)
    ssr_img = zero4 if ssr_img is None else _h(ssr_img)
    refl = zero4 if refl is None else _h(refl)
    if shadow_map is None:
        shadow_map = np.zeros((4, 4), np.float32)
    sm = np.ascontiguousarray(shadow_map, np.float32)
    rt = _h(rt)
    out = np.empty((H, W, 4), np.float16 if out_format == T.VK_FORMAT_R16G16B16A16_SFLOAT else np.uint8)
    a8 = np.ascontiguousarray(albedo, np.uint8)
    d = np.ascontiguousarray(depth, np.float32)
    lib().vo_composition(_p(pfd), W, H, int(shadow_mode), int(ao_mode), int(reflection_mode), _p(a8), _p(_h(normals)), _p(_h(motion)), _p(d),
                         _p(sm), sm.shape[1], sm.shape[0], _p(ssao_img), _p(ssr_img), _p(rt), rt.shape[-1], _p(refl), int(out_format), _p(out))
    return out


def raygen_pixel_rays(pfd, depth, normals, x, y, ao_spp=2):
    """The shadow ray and the `ao_spp` AO rays raygen.rgen generates for pixel (x, y): array [n, 8] (origin, tMin, direction, tMax)."""
    H, W = depth.shape[:2]
    rays = np.zeros((1 + ao_spp, 8), np.float32)
    d = np.ascontiguousarray(depth, np.float32)
    n = lib().vo_raygen_pixel_rays(_p(pfd), W, H, int(x), int(y), _p(d), _p(_h(normals)), int(ao_spp), _p(rays))
    return rays[:n]


class OracleScene:
    def __init__(self, scene):
        v = np.ascontiguousarray(scene.vertices)
        i = np.ascontiguousarray(scene.indices, np.uint32)
        p = np.ascontiguousarray(scene.primitives)
        assert v.dtype == T.Vertex and p.dtype == T.Primitive
        self._s = lib().vo_scene_create(_p(v), len(v), _p(i), len(i), _p(p), len(p))
        for t in getattr(scene, "textures", []):
            self.add_texture(t.rgba, t.format, t.sampler)

    def add_texture(self, rgba8, fmt=T.VK_FORMAT_R8G8B8A8_UNORM, sampler=None):
        """ResourceManager::UploadTextureFromData: returns the texture index. sampler = (mag, min, wrap_u, wrap_v); None = default."""
        a = np.ascontiguousarray(rgba8, np.uint8)
        mag, mn, wu, wv = (1, 1, 0, 0) if sampler is None else [int(x) for x in sampler]
        return lib().vo_scene_add_texture(self._s, a.shape[1], a.shape[0], _p(a), int(fmt), mag, mn, wu, wv)

    def sample_texture(self, idx, u, v):
        out = np.zeros(4, np.float32)
        lib().vo_sample_texture(self._s, int(idx), float(u), float(v), _p(out))
        return out

    def __del__(self):
        if getattr(self, "_s", None):
            lib().vo_scene_destroy(self._s)
            self._s = None

    @property
    def num_triangles(self):
        return lib().vo_scene_num_triangles(self._s)

    def trace_any(self, o, d, tmin, tmax):
        o = np.asarray(o, np.float32); d = np.asarray(d, np.float32)
        return bool(lib().vo_trace_any(self._s, _p(o), _p(d), tmin, tmax))

    def trace_closest(self, o, d, tmin, tmax):
        o = np.asarray(o, np.float32); d = np.asarray(d, np.float32)
        tuv = np.zeros(3, np.float64); gp = np.zeros(2, np.uint32)
        hit = lib().vo_trace_closest(self._s, _p(o), _p(d), tmin, tmax, _p(tuv), _p(gp))
        return (tuv, gp) if hit else None

    def brute_force(self, o, d, tmin, tmax):
        """One ray against every triangle in double precision: (any_hit, closest_t, margin). See vo_brute_force."""
        o = np.ascontiguousarray(o, np.float32); d = np.ascontiguousarray(d, np.float32)
        out = np.zeros(3, np.float64)
        lib().vo_brute_force(self._s, _p(o), _p(d), float(tmin), float(tmax), _p(out))
        return bool(out[0]), float(out[1]), float(out[2])

    def gbuffer(self, pfd, W, H, want_ids=False):
        albedo = np.empty((H, W, 4), np.uint8)
        normals = np.empty((H, W, 4), np.float16)
        motion = np.empty((H, W, 4), np.float16)
        depth = np.empty((H, W), np.float32)
        ids = np.empty((H, W, 2), np.int32) if want_ids else None
        lib().vo_gbuffer(self._s, _p(pfd), W, H, _p(albedo), _p(normals), _p(motion), _p(depth), _p(ids))
        g = dict(albedo=albedo, normals=normals, motion=motion, depth=depth)
        if want_ids:
            g["ids"] = ids
        return g

    def shade_hits(self, pfd, kind, records):
        """The per-hit code of the passes on the given hits, kinds and output words as vhr_debug_shade_hits (Context.shade_hits):
        [n, T.SHADE_OUT_WORDS] uint32."""
        rec = np.ascontiguousarray(records, T.ShadeRecord).reshape(-1)
        out = np.zeros((len(rec), T.SHADE_OUT_WORDS), np.uint32)
        if lib().vo_shade_hits(self._s, _p(pfd), int(kind), _p(rec), len(rec), _p(out)) != 0:
            raise ValueError("vo_shade_hits: unknown kind or a record naming a texture / triangle that does not exist")
        return out

    def raytraced(self, pfd, W, H, alpha_test=False):
        """The fully ray-traced render path's "Raytracing Pass": [H, W, 4] uint8 B8G8R8A8_UNORM "RaytracedOutput"."""
        out = np.empty((H, W, 4), np.uint8)
        lib().vo_raytraced(self._s, _p(pfd), W, H, int(bool(alpha_test)), _p(out))
        return out

    def raygen(self, pfd, depth, normals, ao_spp=2, flags=7, rows=None, want_t=False):
        H, W = depth.shape[:2]
        y0, y1 = (0, H) if rows is None else rows
        sa = np.zeros((H, W, 2), np.float16)
        refl = np.zeros((H, W, 4), np.float16)
        t = np.full((H, W), -1.0, np.float32) if want_t else None
        cnt = C.c_uint64(0)
        d = np.ascontiguousarray(depth, np.float32)
        lib().vo_raygen(self._s, _p(pfd), W, H, y0, y1, ao_spp, flags, _p(d), _p(_h(normals)), _p(sa), _p(refl),
                        _p(t), C.byref(cnt))
        out = dict(shadow_ao=sa, reflections=refl, rays=cnt.value)
        if want_t:
            out["refl_t"] = t
        return out
