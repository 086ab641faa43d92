"""GPU parity: screen-space reflections (ssr.comp through the C-ABI) vs the CPU oracle."""
import os

import numpy as np
import pytest

import helpers as Hh
import checker as O
from vulkanhybridrenderer_b200 import capi, host_api
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu
F4 = T.VK_FORMAT_R16G16B16A16_SFLOAT


def _check(out, ref, what):
    """Bit identity of the fp16 image with the checker's: the march is a chain of threshold tests, every one of them evaluated in the
    oracle's operations and order, so one flipped comparison (a pixel that lands somewhere else entirely) or one ulp in a helper is a
    failure. The found-mask and radiance statistics are printed (and reported on failure) as the diagnosis."""
    o, r = out.astype(np.float32), ref.astype(np.float32)
    fo, fr = o[..., 3] > 0, r[..., 3] > 0
    mask_agree = float(np.mean(fo == fr))
    both = fo & fr
    err = np.abs(o[both][:, :3] - r[both][:, :3]) / np.maximum(1.0, np.abs(r[both][:, :3]))
    ok = float(np.mean(np.all(err <= 2e-3, axis=-1))) if both.any() else 1.0
    same = np.all(out.view(np.uint16) == ref.view(np.uint16), axis=-1)
    exact = float(np.mean(same))
    stats = (f"{what}: found {fr.mean()*100:.1f}% of pixels, mask agreement {mask_agree*100:.4f}%, radiance within 2e-3 {ok*100:.4f}%, "
             f"bit-exact {exact*100:.4f}%")
    print(f"[parity] {stats}")
    assert fr.mean() > 0.02, "degenerate SSR frame"
    assert same.all(), f"{stats}; first differing pixels (y, x): {np.argwhere(~same)[:8].tolist()}"
    return exact


SSR_CASES = [
    pytest.param((320, 184), (25.0, 0.1, 0.5, 10), "default", None, id="size0-params0"),
    pytest.param((203, 117), (6.0, 0.25, 1.0, 4), "default", None, id="size1-params1"),
    pytest.param((96, 64), (8.0, 0.1, 0.5, 0), "default", None, id="size2-params2"),
] + [pytest.param((203, 117), (6.0, 0.25, 1.0, 4), cam, None, id=f"{cam}-203x117") for cam in Hh.CAMERA_CASES[1:]] + [
    # below 16 pixels in one dimension (no step skipping), and dispatches that cover only part of the image
    pytest.param((13, 40), (8.0, 0.1, 0.5, 4), "default", None, id="13x40"),
    pytest.param((45, 9), (8.0, 0.1, 0.5, 4), "jitter", None, id="45x9-jitter"),
    pytest.param((61, 37), (8.0, 0.1, 0.5, 4), "default", (5, 3), id="61x37-partial"),
    pytest.param((203, 117), (6.0, 0.25, 1.0, 4), "finite_far", (20, 14), id="203x117-partial-finite_far"),
]


@pytest.mark.parametrize("size,params,cam,groups", SSR_CASES)
def test_ssr_vs_oracle(size, params, cam, groups):
    """`groups`: the (x, y) workgroup counts of a dispatch that covers only the top-left part of the image (default: all of it);
    the pixels outside it keep what the image held."""
    W, H = size
    sc, osc, pfd, g = Hh.camera_case(cam, W, H)
    xg, yg = groups or (HP.groups(W), HP.groups(H))
    ref = O.ssr(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], *params)
    with capi.Context(W, H) as ctx:
        ctx.update_per_frame_ubo(pfd)
        for name, fmt in Hh.GBUF_IMAGES.items():
            ctx.actualize_image(name, fmt)
        ctx.actualize_image(HP.N_SSR, F4)
        ctx.image_upload(HP.N_ALBEDO, g["albedo"]); ctx.image_upload(HP.N_NORMALS, g["normals"])
        ctx.image_upload(HP.N_MOTION, g["motion"]); ctx.image_upload(HP.N_DEPTH, g["depth"])
        ctx.image_upload(HP.N_SSR, np.full((H, W, 4), 7.0, np.float16))
        ctx.bind_pass_images([HP.N_ALBEDO, HP.N_NORMALS, HP.N_MOTION, HP.N_DEPTH, HP.N_SSR])
        pc = np.array(params, T.SSRPushConstants)
        n0 = ctx.kernel_launches
        ctx.dispatch(HP.SHADER_SSR, xg, yg, 1, pc)
        # the depth quad-image pre-pass + the march (+ the tile pre-pass of the opt-in step skipping)
        assert ctx.kernel_launches == n0 + 2 + (1 if os.environ.get("VHR_SSR_SKIP", "0") not in ("", "0") else 0)
        out = ctx.image_download(HP.N_SSR)
        # push-constant size is checked like the reference's assert (compute_execution_context.h:23)
        with pytest.raises(capi.VhrError):
            ctx.dispatch(HP.SHADER_SSR, xg, yg, 1, np.array([0.75], np.float32))
        # row band: only the band is written (multi-GPU split)
        ctx.image_upload(HP.N_SSR, np.full((H, W, 4), 7.0, np.float16))
        r0, r1 = min(16, H // 3), min(40, 2 * H // 3)
        ctx.set_option(capi.OPT_ROW_BEGIN, r0); ctx.set_option(capi.OPT_ROW_END, r1)
        ctx.dispatch(HP.SHADER_SSR, xg, yg, 1, pc)
        band = ctx.image_download(HP.N_SSR)
    xe, ye = min(W, 8 * xg), min(H, 8 * yg)
    _check(out[:ye, :xe], ref[:ye, :xe], f"ssr {W}x{H} {params} camera {cam}" + (f" dispatch {xg}x{yg} groups" if groups else ""))
    untouched = np.ones((H, W), bool)
    untouched[:ye, :xe] = False
    assert np.all(out[untouched].astype(np.float32) == 7.0), "pixels outside the dispatch were written"
    assert np.all(band[:r0].astype(np.float32) == 7.0) and np.all(band[r1:].astype(np.float32) == 7.0)
    assert np.array_equal(band[r0:r1].view(np.uint16), out[r0:r1].view(np.uint16))


def test_ssr_node_in_host_graph():
    """reflection_mode = SSR registers the "SSR Pass" node (hybrid_render_path.cpp:202-243); composition consumes its image."""
    from vulkanhybridrenderer_b200 import camera, scenes
    W, H = 160, 96
    sc = scenes.sponza_like(12_000, seed=5, width=W, height=H, n_clutter=20)
    seq = camera.FrameSequencer(W, H, sc.light)
    pfd = seq.next(sc.camera)
    with host_api.Renderer(W, H) as r:
        r.load_scene(sc)
        r.set_modes(shadow=0, ao=0, reflection=1, denoise=True)
        r.set_gbuffer_producer(True)
        order = r.execution_order()
        assert "SSR Pass" in order and order.index("SSR Pass") < order.index("Composition Pass")
        r.render(pfd)
        ctx = r.ctx
        g = {k: ctx.image_download(n) for k, n in (("albedo", HP.N_ALBEDO), ("normals", HP.N_NORMALS), ("motion", HP.N_MOTION), ("depth", HP.N_DEPTH))}
        want = O.ssr(pfd, g["albedo"], g["normals"], g["motion"], g["depth"])
        got = ctx.image_download(HP.N_SSR)
        _check(got, want, "host graph ssr")
        out = ctx.image_download(HP.N_RENDER_OUTPUT)
        ref_out = O.composition(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], ctx.image_download(HP.N_DENOISED), 0, 0, 1,
                                ssr_img=got, out_format=T.VK_FORMAT_B8G8R8A8_SRGB)
        code = np.abs(out.astype(np.int32) - ref_out.astype(np.int32))
        assert code.max() <= 1 and np.mean(code == 0) >= 0.995
