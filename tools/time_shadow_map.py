"""Times the CUDA "Shadow Map Pass" (vhr_shadow_map_pass, 4096^2 D32) against the ray-traced alternative (the Raytrace Pass with
shadow rays only, 1080p) on the same scenes: the two shadow techniques of the reference's hybrid path side by side.

    python tools/time_shadow_map.py [--iters 200] [--out profiles/r03/time_shadow_map.json]

Scenes: sponza_like at 260 k and 3 M triangles; the shadow map with the reference's fixed light window (half of the hall lies
beyond its depth-0 plane and is clipped) and with a window fitted to the scene. Device time from timestamps (CUDA events) around
`--iters` back-to-back passes after a warm-up. The map (64 MiB) fits the 126 MB L2, so repeated passes find it there.
Lower bound: 48 B per triangle read from the triangle buffer + 64 MiB written, at 7.7 TB/s (HBM3e, B200 data sheet)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from vulkanhybridrenderer_b200 import camera, capi, scenes  # noqa: E402
from vulkanhybridrenderer_b200 import hybrid_path as HP  # noqa: E402
from vulkanhybridrenderer_b200 import types as T  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:          # the numbers still stand; say that the device could not be named
        return f"unknown ({e})", "unknown"


def timed(ctx, fn, iters, warmup=10):
    for _ in range(warmup):
        fn()
    capi._check(capi.lib().vhr_create_query_pool(ctx._h, 2))
    capi._check(capi.lib().vhr_write_timestamp(ctx._h, 0))
    for _ in range(iters):
        fn()
    capi._check(capi.lib().vhr_write_timestamp(ctx._h, 1))
    ctx.synchronize()
    ms = C.c_double()
    capi._check(capi.lib().vhr_get_query_elapsed_ms(ctx._h, 0, 1, C.byref(ms)))
    return ms.value / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "time_shadow_map.json"))
    ap.add_argument("--triangles", default="260000,3000000")
    a = ap.parse_args()
    name, power = device_info()
    print(f"[time_shadow_map] device {name}, power limit {power}")
    res = dict(device=name, power_limit=power, iters=a.iters, map="4096x4096 D32_SFLOAT", ray_pass="1920x1080, shadow rays only", runs=[])
    S, W, H = 4096, 1920, 1080
    for n in (int(x) for x in a.triangles.split(",")):
        sc = scenes.sponza_like(n, width=W, height=H)
        with capi.Context(W, H) as ctx:
            ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
            n_tris = ctx.bvh_stats().n_triangles
            path = HP.HybridRenderPath(ctx, W, H, composition=T.VK_FORMAT_B8G8R8A8_SRGB, shadow_map_size=(S, S))
            lo, hi = np.array(ctx.bvh_stats().scene_min), np.array(ctx.bvh_stats().scene_max)
            d = sc.light["direction"][:3]
            bound_ms = (48.0 * n_tris + S * S * 4) / HBM_BYTES_PER_S * 1e3
            row = dict(triangles=n_tris, lower_bound_ms=bound_ms)
            for window, pv in (("reference", camera.light_projview(d)), ("fitted", camera.fit_light_projview(d, lo, hi))):
                light = sc.light.copy()
                light["projview"] = pv
                pfd = camera.FrameSequencer(W, H, light).next(sc.camera)
                ctx.update_per_frame_ubo(pfd)
                ms = timed(ctx, path.shadow_map_pass, a.iters)
                covered = float(np.mean(ctx.image_download(HP.N_SHADOW_MAP) > 0))
                row[f"shadow_map_{window}_ms"] = ms
                row[f"shadow_map_{window}_covered"] = covered
                print(f"[time_shadow_map] {n_tris} triangles, {window} window: {ms:.4f} ms per 4096^2 map ({covered*100:.1f}% covered), "
                      f"bound {bound_ms:.4f} ms")
            g = path.gsets[0]
            ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
            ctx.gbuffer_pass(W, H)
            ctx.set_option(capi.OPT_TRACE_AO, 0)
            ctx.set_option(capi.OPT_TRACE_REFLECTIONS, 0)
            row["ray_shadows_1080p_ms"] = timed(ctx, path.raytrace_pass, a.iters)
            print(f"[time_shadow_map] {n_tris} triangles: ray-traced shadows at 1080p {row['ray_shadows_1080p_ms']:.4f} ms")
            res["runs"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
