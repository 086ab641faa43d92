"""Python mirror of the hot-path nodes of HybridRenderPath::RegisterPath, issued call by call through the C-ABI.

Reference: /root/reference/src/render_paths/hybrid_render_path.cpp
    :101-136  "Raytrace Pass"      (TraceRays, bindings 0 normals, 1 depth, 2 shadow/AO, 3 reflections)
    :138-200  "SSAO Pass" + "SSAO Blur Pass"
    :245-331  "SVGF Denoise Pass"  (five persistent storage images, temporal + 5 a-trous dispatches, three blits,
                                    ping-pong swaps; "Denoised" = iteration 3's output, SURVEY Q1)
The C++ twin of this file (host/hybrid_render_path.cpp -> libvhr_host.so) is what a maintainer of the reference links;
this one exists so tests and bench.py can drive exactly the same call sequence from Python. No CPU fallback anywhere:
every call lands in libvhr_b200.so.
"""
import numpy as np

from . import capi
from . import types as T

F4, F2 = T.VK_FORMAT_R16G16B16A16_SFLOAT, T.VK_FORMAT_R16G16_SFLOAT

N_ALBEDO = "Albedo"
N_NORMALS = "World Space Normals and Object IDs"
N_MOTION = "Motion Vectors and Metallic Roughness"
N_DEPTH = "Depth"
N_RT = "Raytraced Shadows and Ambient Occlusion"
N_REFL = "Raytraced Reflections"
N_DENOISED = "Denoised Raytraced Shadows and Ambient Occlusion"
N_SSAO_RAW = "Screen Space Ambient Occlusion Raw"
N_SSAO = "Screen Space Ambient Occlusion"
N_SSR = "Screen Space Reflections"
N_SHADOW_MAP = "Shadow Map"
N_RENDER_OUTPUT = "RENDER_OUTPUT"

GBUFFER_FORMATS = {N_ALBEDO: T.VK_FORMAT_B8G8R8A8_UNORM, N_NORMALS: F4, N_MOTION: F4, N_DEPTH: T.VK_FORMAT_D32_SFLOAT}

SHADER_SVGF = "hybrid_render_path/svgf.comp"
SHADER_ATROUS = "hybrid_render_path/svgf_atrous_filter.comp"
SHADER_SSAO = "hybrid_render_path/ssao.comp"
SHADER_SSAO_BLUR = "hybrid_render_path/ssao_blur.comp"
SHADER_SSR = "hybrid_render_path/ssr.comp"
SHADER_COMPOSITION = "hybrid_render_path/composition.frag"

# common.glsl:12-25 / hybrid_render_path.h:4-20
SHADOW_MODE_RAYTRACED, SHADOW_MODE_RASTERIZED, SHADOW_MODE_OFF = 0, 1, 2
AO_MODE_RAYTRACED, AO_MODE_SSAO, AO_MODE_OFF = 0, 1, 2
REFLECTION_MODE_RAYTRACED, REFLECTION_MODE_SSR, REFLECTION_MODE_OFF = 0, 1, 2

# per-pixel algorithmic bytes (SURVEY §8d / DESIGN.md): each distinct texel once
BYTES_TEMPORAL = 52
BYTES_ATROUS = 24
BYTES_BLIT = 16
BYTES_RAYGEN_IO = 12 + 4          # depth + normals in, RG16F out (reflections add 8)
BYTES_SSAO = 20
BYTES_SSAO_BLUR = 16
BYTES_SSR = 4 + 8 + 4 + 8 + 8     # compulsory G-buffer in (depth 4, normals 8, albedo 4, motion 8) + RGBA16F out 8
BYTES_COMPOSITION = 4 + 8 + 8 + 4 + 8 + 4   # albedo, normals, motion texel, depth, denoised shadow/AO in; BGRA8 out (+8 reflections)


def groups(n):
    return n // 8 + (n % 8 != 0)       # hybrid_render_path.cpp:291-294


class HybridRenderPath:
    """Owns the images of the hot-path passes on one context and replays the reference's per-frame call sequence."""

    def __init__(self, ctx, width, height, gbuffer_sets=1, ssao=False, composition=None, shadow_map_size=(4096, 4096), rt_sets=1, svgf_fused=False,
                 blit_alias=None):
        """composition: None (no composition pass) or the VkFormat of RENDER_OUTPUT (B8G8R8A8_SRGB = the reference's
        swapchain; R16G16B16A16_SFLOAT = linear HDR radiance for parity measurements)."""
        self.ctx, self.W, self.H = ctx, width, height
        # B200 modes of the SVGF node (HybridRenderPath::svgf_fused of host/hybrid_render_path.h): the call sequence below stays the
        # reference's; the library fuses svgf.comp with a-trous iteration 0 and turns the three blits into copy-on-write aliases
        ctx.set_option(capi.OPT_SVGF_FUSED, int(bool(svgf_fused)))
        ctx.set_option(capi.OPT_BLIT_ALIAS, int(bool(svgf_fused if blit_alias is None else blit_alias)))
        self.gsets = []
        for s in range(gbuffer_sets):
            sfx = "" if s == 0 else f" [{s}]"
            names = {k: k + sfx for k in GBUFFER_FORMATS}
            for k, n in names.items():
                ctx.actualize_image(n, GBUFFER_FORMATS[k])
            self.gsets.append(names)
        # rt_sets = 2 (multi-GPU fused partition): the ray pass of frame k+1 stores into OTHER ranks' images while those may
        # still be reading frame k's, so consecutive frames alternate between two output sets
        self.rt_sets = []
        for s in range(rt_sets):
            sfx = "" if s == 0 else f" [{s}]"
            ctx.actualize_image(N_RT + sfx, F2)
            ctx.actualize_image(N_REFL + sfx, F4)
            self.rt_sets.append((N_RT + sfx, N_REFL + sfx))
        ctx.actualize_image(N_DENOISED, F4)
        if ssao or composition is not None:
            ctx.actualize_image(N_SSAO_RAW, F4)
            ctx.actualize_image(N_SSAO, F4)
        if composition is not None:      # hybrid_render_path.cpp:335-349: every sampled input exists even when its mode is off
            ctx.actualize_image(N_SSR, F4)
            ctx.actualize_image(N_SHADOW_MAP, T.VK_FORMAT_D32_SFLOAT, *shadow_map_size)
            ctx.actualize_image(N_RENDER_OUTPUT, composition)
        # hybrid_render_path.cpp:247-261
        pc = np.zeros((), T.SVGFPushConstants)
        pc["integrated_shadow_and_ao"] = (ctx.upload_new_storage_image(width, height, F4),
                                          ctx.upload_new_storage_image(width, height, F4))
        pc["prev_frame_normals_and_object_ids"] = ctx.upload_new_storage_image(width, height, F4)
        pc["shadow_and_ao_history"] = ctx.upload_new_storage_image(width, height, F4)
        pc["shadow_and_ao_moments_history"] = ctx.upload_new_storage_image(width, height, F2)
        self.pc = pc
        self.ssao_radius = np.array(0.75, np.float32)
        # hybrid_render_path.cpp:203-208
        self.ssr_pc = np.array((25.0, 0.1, 0.5, 10), T.SSRPushConstants)
        self.timestamps = None

    # ---- optional per-pass timestamps (render_graph.cpp:167-182) --------------------------------------------------
    PASS_LABELS = ("raytrace", "svgf_temporal", "atrous0", "atrous1", "atrous2", "atrous3", "atrous4", "blits")

    def enable_timestamps(self, frames):
        """Query pool with len(PASS_LABELS)+1 timestamps per frame for `frames` frames."""
        self._ts_per_frame = len(self.PASS_LABELS) + 1
        capi._check(capi.lib().vhr_create_query_pool(self.ctx._h, self._ts_per_frame * frames))
        self.timestamps = 0

    def _stamp(self):
        if self.timestamps is not None:
            capi._check(capi.lib().vhr_write_timestamp(self.ctx._h, self.timestamps))
            self.timestamps += 1

    def pass_times_ms(self, frames):
        """Per-pass device time (ms) of each recorded frame: array [frames, len(PASS_LABELS)]."""
        import ctypes as C
        out = np.zeros((frames, len(self.PASS_LABELS)))
        ms = C.c_double()
        for f in range(frames):
            b = f * self._ts_per_frame
            for k in range(len(self.PASS_LABELS)):
                capi._check(capi.lib().vhr_get_query_elapsed_ms(self.ctx._h, b + k, b + k + 1, C.byref(ms)))
                out[f, k] = ms.value
        return out

    # ---- passes ---------------------------------------------------------------------------------------------------
    def raytrace_pass(self, gset=0, rtset=0):
        g = self.gsets[gset]
        with self.ctx.debug_label("Raytrace Pass"):
            self.ctx.bind_pass_images([g[N_NORMALS], g[N_DEPTH], *self.rt_sets[rtset]])
            self.ctx.trace_rays(self.W, self.H)

    def ssao_passes(self, gset=0):
        g = self.gsets[gset]
        gx, gy = groups(self.W), groups(self.H)
        self.ctx.bind_pass_images([g[N_NORMALS], g[N_DEPTH], N_SSAO_RAW])     # hybrid_render_path.cpp:143-150
        # the reference dispatches ssao.comp WITHOUT push constants (Q15) => radius 0.75 unless the caller set one
        self.ctx.dispatch(SHADER_SSAO, gx, gy, 1, self.ssao_radius)
        self.ctx.bind_pass_images([N_SSAO_RAW, N_SSAO])
        self.ctx.dispatch(SHADER_SSAO_BLUR, gx, gy, 1, self.ssao_radius)

    def ssr_pass(self, gset=0):
        """"SSR Pass", hybrid_render_path.cpp:202-243: 0 albedo, 1 normals, 2 motion / metallic-roughness, 3 depth, 4 output."""
        g = self.gsets[gset]
        self.ctx.bind_pass_images([g[N_ALBEDO], g[N_NORMALS], g[N_MOTION], g[N_DEPTH], N_SSR])
        self.ctx.dispatch(SHADER_SSR, groups(self.W), groups(self.H), 1, self.ssr_pc)

    def svgf_denoise_pass(self, gset=0, rtset=0):
        with self.ctx.debug_label("SVGF Denoise Pass"):
            self._svgf_denoise_body(gset, rtset)

    def _svgf_denoise_body(self, gset=0, rtset=0):
        """hybrid_render_path.cpp:288-330, statement by statement."""
        ctx, pc, g = self.ctx, self.pc, self.gsets[gset]
        gx, gy = groups(self.W), groups(self.H)
        ctx.bind_pass_images([g[N_NORMALS], g[N_MOTION], g[N_DEPTH], self.rt_sets[rtset][0], N_DENOISED])
        ctx.dispatch(SHADER_SVGF, gx, gy, 1, pc)
        self._stamp()
        for i in range(5):
            pc["atrous_step"] = 1 << i
            ctx.dispatch(SHADER_ATROUS, gx, gy, 1, pc)
            if i == 0:
                ctx.blit_storage_to_storage(int(pc["integrated_shadow_and_ao"][1]), int(pc["shadow_and_ao_history"]))
            pc["integrated_shadow_and_ao"] = pc["integrated_shadow_and_ao"][::-1].copy()
            self._stamp()
        ctx.blit_transient_to_storage(g[N_NORMALS], int(pc["prev_frame_normals_and_object_ids"]))
        ctx.blit_storage_to_transient(int(pc["integrated_shadow_and_ao"][1]), N_DENOISED)
        pc["integrated_shadow_and_ao"] = pc["integrated_shadow_and_ao"][::-1].copy()
        self._stamp()

    def gbuffer_pass(self, gset=0):
        """"G-Buffer Pass", hybrid_render_path.cpp:13-56: G-buffer set `gset` (0 albedo, 1 normals/ids, 2 motion/metallic-roughness,
        3 depth) produced by primary rays for the per-frame constants last uploaded. Under a fused partition whose G-buffer sets are
        exchanged (multi_gpu.setup_fused_partition(..., exchange_gbuffer=True)) every rank traces its own rows and ends with the whole
        G-buffer."""
        g = self.gsets[gset]
        with self.ctx.debug_label("G-Buffer Pass"):
            self.ctx.bind_pass_images([g[N_ALBEDO], g[N_NORMALS], g[N_MOTION], g[N_DEPTH]])
            self.ctx.gbuffer_pass(self.W, self.H)

    def shadow_map_pass(self):
        """"Shadow Map Pass", hybrid_render_path.cpp:58-99: the Shadow Map as depth attachment 0, rasterised from the light."""
        with self.ctx.debug_label("Shadow Map Pass"):
            self.ctx.bind_pass_images([N_SHADOW_MAP])
            self.ctx.shadow_map_pass()

    def composition_pass(self, shadow_mode=SHADOW_MODE_RAYTRACED, ao_mode=AO_MODE_RAYTRACED, reflection_mode=REFLECTION_MODE_OFF,
                         denoised=True, gset=0):
        """hybrid_render_path.cpp:333-379: nine sampled inputs by binding, RENDER_OUTPUT as colour attachment 0, Draw(3,1,0,0)."""
        g = self.gsets[gset]
        self.ctx.bind_pass_images([g[N_ALBEDO], g[N_NORMALS], g[N_MOTION], g[N_DEPTH], N_SHADOW_MAP, N_SSAO, N_SSR,
                                   N_DENOISED if denoised else N_RT, N_REFL, N_RENDER_OUTPUT])
        self.ctx.draw(SHADER_COMPOSITION, (shadow_mode, ao_mode, reflection_mode))

    # semaphores of frame_overlapped, per ray-output set p: the set may be overwritten / the set has been written
    SEM_RT_SET_FREE, SEM_RT_SET_WRITTEN = (0, 1), (2, 3)

    def frame_overlapped(self, pfd, k, gset=0):
        """frame() with two frames in flight (needs rt_sets=2): the Raytrace Pass of frame k is recorded on queue 1 into ray-output
        set k & 1 and only waits for the consumers of that set two frames ago, so it runs under the SVGF Denoise Pass of frame k-1,
        which is still executing on queue 0. Same kernels, same inputs, same images as frame(): only the schedule differs.
        The caller keeps the G-buffer of frame k in a set that frame k-1 does not use (gbuffer_sets=2, gset=k & 1) and reads the
        results of frame k on queue 0 (selected on return) before calling this for frame k+1... or any time before frame k+2."""
        ctx, p = self.ctx, k & 1
        assert len(self.rt_sets) >= 2, "frame_overlapped needs rt_sets=2"
        # everything recorded on queue 0 so far — frame k-1's denoiser and whatever read its images — is what frame k+1's ray pass
        # (which overwrites set (k-1) & 1) has to wait for
        ctx.select_queue(0)
        ctx.queue_signal(self.SEM_RT_SET_FREE[p ^ 1])
        ctx.select_queue(1)
        ctx.queue_wait(self.SEM_RT_SET_FREE[p])
        ctx.update_per_frame_ubo(pfd)
        self.raytrace_pass(gset, p)
        ctx.queue_signal(self.SEM_RT_SET_WRITTEN[p])
        ctx.select_queue(0)
        ctx.queue_wait(self.SEM_RT_SET_WRITTEN[p])
        self.svgf_denoise_pass(gset, p)

    def frame(self, pfd, gset=0, rtset=0):
        """Raytrace Pass -> SVGF Denoise Pass for one frame whose G-buffer already sits in image set `gset`."""
        self.ctx.update_per_frame_ubo(pfd)
        self._stamp()
        self.raytrace_pass(gset, rtset)
        self._stamp()
        self.svgf_denoise_pass(gset, rtset)
