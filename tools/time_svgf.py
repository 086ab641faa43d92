"""Quick device timing of the SVGF / SSAO kernels through the C-ABI (development aid, not the bench)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np
from vulkanhybridrenderer_b200 import capi, types as T

F4, F2 = T.VK_FORMAT_R16G16B16A16_SFLOAT, T.VK_FORMAT_R16G16_SFLOAT


def elapsed(ctx, a, b):
    ms = C.c_double()
    capi._check(capi.lib().vhr_get_query_elapsed_ms(ctx._h, a, b, C.byref(ms)))
    return ms.value


def main(W=1920, H=1080, reps=20):
    rng = np.random.default_rng(0)
    pfd = np.zeros((), T.PerFrameData)
    pfd["display_size"] = (W, H); pfd["display_size_inverse"] = (1.0 / W, 1.0 / H); pfd["frame_index"] = 3
    pfd["camera_proj_inverse"] = np.eye(4); pfd["camera_view"] = np.eye(4)
    normals = np.zeros((H, W, 4), np.float16)
    n = rng.standard_normal((H // 40 + 1, W // 40 + 1, 3)); n /= np.linalg.norm(n, axis=-1, keepdims=True)
    normals[..., :3] = np.kron(n, np.ones((40, 40, 1)))[:H, :W]
    normals[..., 3] = np.kron(rng.integers(0, 200, (H // 40 + 1, W // 40 + 1)), np.ones((40, 40)))[:H, :W]
    integ = np.empty((H, W, 4), np.float16)
    integ[..., 0] = rng.integers(0, 2, (H, W)); integ[..., 1] = rng.integers(0, 3, (H, W)) * 0.5
    integ[..., 2:] = rng.uniform(0, 0.25, (H, W, 2))
    with capi.Context(W, H) as ctx:
        # with a second queue every a-trous dispatch launches at once: a deferred one would be dropped by the next dispatch's overwrite
        ctx.select_queue(1); ctx.select_queue(0)
        ctx.update_per_frame_ubo(pfd)
        ctx.actualize_image("n", F4); ctx.image_upload("n", normals)
        a, b = ctx.upload_new_storage_image(W, H, F4), ctx.upload_new_storage_image(W, H, F4)
        ctx.storage_image_upload(a, integ)
        ctx.bind_pass_images(["n"])
        capi._check(capi.lib().vhr_create_query_pool(ctx._h, 2))
        gx, gy = (W + 7) // 8, (H + 7) // 8
        for variant in [int(v) for v in os.environ.get("VHR_TIME_VARIANTS", "1,2,3").split(",")]:
            ctx.set_option(capi.OPT_ATROUS_VARIANT, variant)
            for step in (1, 2, 4, 8, 16):
                pc = np.zeros((), T.SVGFPushConstants); pc["integrated_shadow_and_ao"] = (a, b); pc["atrous_step"] = step
                for _ in range(3):
                    ctx.dispatch("hybrid_render_path/svgf_atrous_filter.comp", gx, gy, 1, pc)
                capi.lib().vhr_write_timestamp(ctx._h, 0)
                for _ in range(reps):
                    ctx.dispatch("hybrid_render_path/svgf_atrous_filter.comp", gx, gy, 1, pc)
                capi.lib().vhr_write_timestamp(ctx._h, 1)
                us = elapsed(ctx, 0, 1) / reps * 1e3
                print(f"atrous variant {variant} step {step:2d}: {us:8.1f} us  {W*H*24/us/1e3:8.1f} GB/s algorithmic")


if __name__ == "__main__":
    main(*(int(x) for x in sys.argv[1:]))
