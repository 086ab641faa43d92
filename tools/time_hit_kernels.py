"""Device timing of the kernels that run the per-hit shading code: gbuffer_kernel<false> (vhr_gbuffer_pass), gbuffer_kernel<true> (the same
pass under an in-process partition of two ranks on one GPU), raytraced_kernel<false> / <true> (the fully ray-traced path's "Raytracing
Pipeline"). One JSON line per run. VHR_LIB_PATH selects the library, so two builds can be compared in alternation:

    for lib in a.so b.so a.so b.so; do VHR_LIB_PATH=$lib python tools/time_hit_kernels.py; done
"""
import ctypes as C
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import multi_gpu as MG
from vulkanhybridrenderer_b200 import types as T


def _events_ms(ctx, fn, reps):
    fn()                                                     # warm-up
    capi.lib().vhr_write_timestamp(ctx._h, 0)
    for _ in range(reps):
        fn()
    capi.lib().vhr_write_timestamp(ctx._h, 1)
    ms = C.c_double()
    capi._check(capi.lib().vhr_get_query_elapsed_ms(ctx._h, 0, 1, C.byref(ms)))
    return ms.value / reps


def main(W=1920, H=1080, tris=260_000, reps=50):
    sc = scenes.add_procedural_textures(scenes.sponza_like(tris, width=W, height=H))
    pfd = camera.FrameSequencer(W, H, sc.light).next(sc.camera)
    out = dict(lib=os.path.basename(capi.LIB_PATH), W=W, H=H, triangles=sc.num_triangles, reps=reps)
    with capi.Context(W, H) as ctx:
        ctx.load_scene(sc)
        ctx.update_per_frame_ubo(pfd)
        capi._check(capi.lib().vhr_create_query_pool(ctx._h, 2))
        gb = [HP.N_ALBEDO, HP.N_NORMALS, HP.N_MOTION, HP.N_DEPTH]
        for n, f in zip(gb, (T.VK_FORMAT_B8G8R8A8_UNORM, T.VK_FORMAT_R16G16B16A16_SFLOAT, T.VK_FORMAT_R16G16B16A16_SFLOAT, T.VK_FORMAT_D32_SFLOAT)):
            ctx.actualize_image(n, f)
        ctx.bind_pass_images(gb)
        out["gbuffer_kernel<false>_ms"] = _events_ms(ctx, lambda: ctx.gbuffer_pass(W, H), reps)
        ctx.actualize_image("RaytracedOutput", T.VK_FORMAT_B8G8R8A8_UNORM)
        ctx.bind_pass_images(["RaytracedOutput"])
        for alpha in (False, True):
            ctx.set_option(capi.OPT_RAYTRACED_ALPHA_TEST, int(alpha))
            out[f"raytraced_kernel<{str(alpha).lower()}>_ms"] = _events_ms(ctx, lambda: ctx.trace_rays(W, H, "Raytracing Pipeline"), reps)
    # gbuffer_kernel<true>: two ranks of one process on one GPU; host clock around the pass of both ranks, ended by a synchronise
    ranks = []
    try:
        for _ in range(2):
            c = capi.Context(W, H)
            c.load_scene(sc)
            ranks.append((c, HP.HybridRenderPath(c, W, H)))
        MG.setup_fused_partition_inprocess([c for c, _ in ranks], [p for _, p in ranks], ray_block_rows=8, exchange_gbuffer=True)

        def both():
            for c, p in ranks:
                c.update_per_frame_ubo(pfd)
                p.gbuffer_pass()
        both()
        for c, _ in ranks:
            c.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            both()
        for c, _ in ranks:
            c.synchronize()
        out["gbuffer_kernel<true>_world2_wall_ms"] = (time.perf_counter() - t0) * 1e3 / reps
    finally:
        for c, _ in ranks:
            c.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main(*(int(x) for x in sys.argv[1:]))
