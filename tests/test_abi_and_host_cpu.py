"""CPU tests: the C-ABI library loads and exports exactly what include/vhr_b200.h declares, fails loudly without a GPU,
and the C++ host (RenderGraph / HybridRenderPath mirrors) schedules passes like the reference.

No compute is issued here: contexts are created with VHR_DEVICE_NONE (validation only)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from vulkanhybridrenderer_b200 import capi, host_api
from vulkanhybridrenderer_b200 import types as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "vhr_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vhr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    L = capi.lib()
    declared = _header_symbols()
    assert len(declared) >= 30
    for s in declared:
        assert hasattr(L, s), f"libvhr_b200.so does not export {s}"
    assert sorted(capi.SYMBOLS) == declared, "capi.SYMBOLS is out of sync with include/vhr_b200.h"


def test_host_library_exports():
    L = host_api.lib()
    for s in host_api.SYMBOLS:
        assert hasattr(L, s)


@pytest.mark.skipif(pytest.importorskip("conftest").HAS_GPU, reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_without_gpu():
    with pytest.raises(capi.VhrError) as e:
        capi.Context(64, 64)
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


def test_validation_context_tables_and_loud_failures():
    F4 = T.VK_FORMAT_R16G16B16A16_SFLOAT
    with capi.Context(64, 48, device=host_api.DEVICE_NONE) as ctx:
        ctx.actualize_image("Depth", T.VK_FORMAT_D32_SFLOAT)
        ctx.actualize_image("Depth", T.VK_FORMAT_D32_SFLOAT)            # same declaration again: fine
        with pytest.raises(capi.VhrError):                                # re-declared with another format (SanityCheck)
            ctx.actualize_image("Depth", F4)
        with pytest.raises(capi.VhrError):
            ctx.actualize_image("Bad", 12345)
        # storage slots: first free slot, reuse after destroy (resource_manager.cpp:866-878)
        a, b, c = (ctx.upload_new_storage_image(64, 48, F4) for _ in range(3))
        assert (a, b, c) == (0, 1, 2)
        ctx.destroy_storage_image(b)
        assert ctx.upload_new_storage_image(64, 48, F4) == 1
        with pytest.raises(capi.VhrError):
            ctx.destroy_storage_image(99)
        # anything that needs the GPU fails loudly
        pc = np.zeros((), T.SVGFPushConstants)
        ctx.update_per_frame_ubo(np.zeros((), T.PerFrameData))
        for call in (lambda: ctx.dispatch("hybrid_render_path/svgf.comp", 8, 6, 1, pc), lambda: ctx.trace_rays(64, 48),
                     lambda: ctx.image_upload("Depth", np.zeros((48, 64), np.float32)),
                     lambda: ctx.shade_hits(T.SHADE_GBUFFER, np.zeros(2, T.ShadeRecord))):
            with pytest.raises(capi.VhrError) as e:
                call()
            assert "VHR_DEVICE_NONE" in str(e.value)
        # slot exhaustion (resource_manager.h:13: 2048 global resources)
        n = 3
        with pytest.raises(capi.VhrError) as e:
            while True:
                ctx.upload_new_storage_image(8, 8, F4)
                n += 1
        assert n == 2048 and "No free storage image slots" in str(e.value)


def test_shade_hits_arguments_are_validated():
    """vhr_debug_shade_hits: an unknown kind or a NULL array is VHR_ERR_INVALID before the device is needed; every kind fails loudly
    on a validation-only context."""
    with capi.Context(8, 8, device=host_api.DEVICE_NONE) as ctx:
        rec = np.zeros(3, T.ShadeRecord)
        for bad in (-1, T.SHADE_ANYHIT_ALPHA + 1, 1 << 20):
            with pytest.raises(capi.VhrError, match="status -1:.*kind"):
                ctx.shade_hits(bad, rec)
        with pytest.raises(capi.VhrError, match="status -1:.*NULL"):
            capi._check(capi.lib().vhr_debug_shade_hits(ctx._h, T.SHADE_TEXTURE, None, 3, capi._ptr(np.zeros(24, np.uint32))))
        for kind in range(T.SHADE_ANYHIT_ALPHA + 1):
            with pytest.raises(capi.VhrError, match="status -2:.*VHR_DEVICE_NONE"):
                ctx.shade_hits(kind, rec)


def test_per_frame_ubo_size_is_checked():
    with capi.Context(8, 8, device=host_api.DEVICE_NONE) as ctx:
        with pytest.raises(capi.VhrError):
            capi._check(capi.lib().vhr_update_per_frame_ubo(ctx._h, capi._ptr(np.zeros(10, np.uint8)), 10))


# ---- render-graph scheduling (render_graph.cpp:686-720) ---------------------------------------------------------------
G, RT, SVGF, COMP = "G-Buffer Pass", "Raytrace Pass", "SVGF Denoise Pass", "Composition Pass"


@pytest.mark.parametrize("modes,want", [
    (dict(shadow=0, ao=2, reflection=2, denoise=False), [G, RT, COMP]),                       # reference defaults (hybrid_render_path.h:32-35)
    (dict(shadow=0, ao=0, reflection=0, denoise=True), [G, RT, SVGF, COMP]),                  # SURVEY §3.2 order
    (dict(shadow=0, ao=1, reflection=2, denoise=True), [G, "SSAO Pass", "SSAO Blur Pass", RT, SVGF, COMP]),
    (dict(shadow=1, ao=0, reflection=2, denoise=True), [G, "Shadow Map Pass", SVGF, COMP]),   # Q21: the else-if drops the ray pass but SVGF still runs (on an unwritten image)
    (dict(shadow=2, ao=2, reflection=2, denoise=True), [G, COMP]),
    (dict(shadow=0, ao=0, reflection=1, denoise=True), [G, "SSR Pass", RT, SVGF, COMP]),      # hybrid_render_path.cpp:202-243
    (dict(shadow=2, ao=2, reflection=1, denoise=False), [G, "SSR Pass", COMP]),
])
def test_execution_order_matches_reference_algorithm(modes, want):
    with host_api.Renderer(128, 72, device=host_api.DEVICE_NONE) as r:
        r.set_modes(**modes)
        got = r.execution_order()
        assert sorted(got) == sorted(want), got
        # dependencies precede consumers; the RENDER_OUTPUT writer is last
        assert got[-1] == COMP and got[0] == G
        if RT in got and SVGF in got:
            assert got.index(RT) < got.index(SVGF)
        if "SSAO Pass" in got:
            assert got.index("SSAO Pass") < got.index("SSAO Blur Pass")


def test_raytraced_path_graph():
    """raytraced_render_path.cpp:11-78: two nodes; switching between the render paths re-registers the nodes."""
    with host_api.Renderer(128, 72, device=host_api.DEVICE_NONE) as r:
        r.set_raytraced_path(False)
        assert r.execution_order() == ["Raytracing Pass", "Composition Pass"]
        r.set_raytraced_path(True)                                   # Rebuild() with the alpha-tested pipeline
        assert r.execution_order() == ["Raytracing Pass", "Composition Pass"]
        r.set_modes(shadow=0, ao=0, reflection=0, denoise=True)
        assert r.execution_order() == [G, RT, SVGF, COMP]
        r.set_raytraced_path(False)
        assert r.execution_order() == ["Raytracing Pass", "Composition Pass"]


def test_rebuild_recreates_svgf_storage_images():
    with host_api.Renderer(128, 72, device=host_api.DEVICE_NONE) as r:
        r.set_modes(shadow=0, ao=0, reflection=2, denoise=True)
        pc = r.svgf_push_constants()
        assert list(pc["integrated_shadow_and_ao"]) == [0, 1] and int(pc["shadow_and_ao_moments_history"]) == 4
        r.set_modes(shadow=0, ao=0, reflection=2, denoise=True)          # Rebuild: Deregister frees the five slots, Register takes them again
        pc2 = r.svgf_push_constants()
        assert list(pc2["integrated_shadow_and_ao"]) == [0, 1]
        # rendering needs the GPU: fails loudly on the validation context, never falls back
        with pytest.raises(capi.VhrError):
            r.render(np.zeros((), T.PerFrameData))


# ---- multi-GPU partition (include/vhr_b200.h, "one frame over several GPUs"): argument validation needs no GPU -------------
def test_partition_arguments_are_validated():
    from vulkanhybridrenderer_b200 import multi_gpu as MG
    H = 1080
    with capi.Context(1920, H, device=host_api.DEVICE_NONE) as ctx:
        bands = [MG.band_rows(H, 4, r)[0] for r in range(4)] + [H]
        ctx.set_partition(4, 1, bands)                                     # well formed
        assert ctx.get_option(capi.OPT_ROW_BEGIN) == bands[1] and ctx.get_option(capi.OPT_ROW_END) == bands[2]
        ctx.clear_partition()
        with pytest.raises(capi.VhrError):
            ctx.set_partition(4, 4, bands)                                 # rank out of range
        with pytest.raises(capi.VhrError):
            ctx.set_partition(9, 0, list(range(0, 1081, 120)))             # more ranks than VHR_MAX_RANKS
        with pytest.raises(capi.VhrError):
            ctx.set_partition(4, 0, bands[:-1] + [H - 8])                  # bands do not cover the image
        with pytest.raises(capi.VhrError):
            ctx.set_partition(4, 0, [0, 30, 540, 810, H])                  # a band thinner than the widest halo
        with pytest.raises(capi.VhrError):
            ctx.set_partition(4, 0, bands, ray_block_rows=4)               # the ray kernel deals 8-row blocks
        with pytest.raises(capi.VhrError):
            ctx.set_partition(4, 0, bands, motion_halo=200)
        # exporting / attaching peer memory needs the device: loud failure, no fallback
        ctx.actualize_image("Depth", T.VK_FORMAT_D32_SFLOAT)
        for call in (lambda: ctx.image_export_ipc("Depth"), lambda: ctx.sync_export_ipc(),
                     lambda: ctx.image_attach_peer("Depth", 1, b"\0" * 64)):
            with pytest.raises(capi.VhrError) as e:
                call()
            assert "VHR_DEVICE_NONE" in str(e.value)


def test_queue_and_semaphore_arguments_are_validated():
    """vhr_select_queue / vhr_queue_signal / vhr_queue_wait: argument checks work without a device; on a validation-only context the
    calls themselves record nothing and succeed."""
    with capi.Context(64, 48, device=host_api.DEVICE_NONE) as ctx:
        ctx.select_queue(0); ctx.select_queue(1); ctx.select_queue(0)
        ctx.queue_signal(0); ctx.queue_wait(0); ctx.queue_wait(capi.MAX_SEMAPHORES - 1)
        for bad in (-1, 2):
            with pytest.raises(capi.VhrError):
                ctx.select_queue(bad)
        for bad in (-1, capi.MAX_SEMAPHORES):
            with pytest.raises(capi.VhrError):
                ctx.queue_signal(bad)
            with pytest.raises(capi.VhrError):
                ctx.queue_wait(bad)
