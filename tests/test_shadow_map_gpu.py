"""GPU: the CUDA "Shadow Map Pass" (vhr_shadow_map_pass) bit for bit against the CPU port (shadow_map_lib.shadow_map), checked
independently through the BVH, end to end through the C++ host, against the ray-traced shadows, and under a partition."""
import numpy as np
import pytest

import checker as O
import helpers as Hh
import shadow_map_lib as SM
from vulkanhybridrenderer_b200 import camera, capi, host_api, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import multi_gpu as MG
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu
D32 = T.VK_FORMAT_D32_SFLOAT


def _fitted(sc):
    p = Hh.world_triangles(sc).reshape(-1, 3)
    return camera.fit_light_projview(sc.light["direction"][:3], p.min(0), p.max(0))


def _pfd(sc, projview, W=64, H=48):
    light = sc.light.copy()
    light["projview"] = projview
    return camera.FrameSequencer(W, H, light).next(sc.camera)


def _render(ctx, pfd, S, name="Shadow Map"):
    ctx.update_per_frame_ubo(pfd)
    ctx.bind_pass_images([name])
    ctx.shadow_map_pass()
    return ctx.image_download(name)


def _assert_bits(got, want, what):
    bad = int(np.sum(got.view(np.uint32) != want.view(np.uint32)))
    print(f"[shadow map] {what}: {bad} of {want.size} texels differ, {int(np.sum(want > 0))} covered")
    assert bad == 0, what


@pytest.mark.parametrize("size", [(64, 64), (100, 37), (256, 256), (1000, 1000)])
@pytest.mark.parametrize("window", ["reference", "fitted"])
def test_tiny_scene_bit_identical(size, window):
    W, H = size
    sc = scenes.tiny_scene()
    pv = camera.light_projview(sc.light["direction"][:3]) if window == "reference" else _fitted(sc)
    pfd = _pfd(sc, pv)
    want = SM.shadow_map(sc, pfd, W, H)
    with capi.Context(64, 48) as ctx:
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.actualize_image("Shadow Map", D32, W, H)
        n0 = ctx.kernel_launches
        _assert_bits(_render(ctx, pfd, W), want, f"tiny {W}x{H} {window}")
        assert ctx.kernel_launches - n0 == 5


def test_sponza_4096_bit_identical_repeatable_queue1_alias():
    sc = scenes.sponza_like(260_000)
    S = 4096
    with capi.Context(64, 48) as ctx:
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.actualize_image("Shadow Map", D32, S, S)
        ctx.actualize_image("Other", D32, S, S)
        for window, pv in (("reference", camera.light_projview(sc.light["direction"][:3])), ("fitted", _fitted(sc))):
            pfd = _pfd(sc, pv)
            want = SM.shadow_map(sc, pfd, S, S)
            _assert_bits(_render(ctx, pfd, S), want, f"sponza 260k {window}")
            _assert_bits(_render(ctx, pfd, S), want, f"sponza 260k {window}, second run")
            ctx.select_queue(1)
            _assert_bits(_render(ctx, pfd, S), want, f"sponza 260k {window}, queue 1")
            ctx.synchronize()
            ctx.select_queue(0)
        # copy-free blits: the map first shares its buffer with another image, then the pass writes it
        ctx.set_option(capi.OPT_BLIT_ALIAS, 1)
        slot = ctx.upload_new_storage_image(S, S, D32)
        ctx.blit_transient_to_storage("Other", slot)
        ctx.blit_storage_to_transient(slot, "Shadow Map")
        _assert_bits(_render(ctx, pfd, S), want, "sponza 260k fitted, after an aliasing blit")
        assert not ctx.storage_image_download(slot).any()        # the blit's source kept its own (zero) texels


def test_depth_through_the_bvh():
    """Orthographic closest-hit rays from the light's depth-1 plane through sampled texel centres (vhr_trace_explicit): the depth
    of the hit agrees with the map; hit / miss agrees with covered / cleared except where the ray grazes an edge."""
    sc = scenes.sponza_like(260_000)
    S, n = 4096, 100_000
    pv = _fitted(sc)
    M = np.asarray(pv, np.float64).T                          # row-major projview
    inv = np.linalg.inv(M)
    rng = np.random.default_rng(7)
    px, py = rng.integers(0, S, n), rng.integers(0, S, n)
    ndc = np.stack([(px + 0.5) / S * 2 - 1, (py + 0.5) / S * 2 - 1, np.ones(n), np.ones(n)], 1)
    o = ndc @ inv.T
    d = (np.array([0, 0, 0, 0.0]) - np.array([0, 0, 1, 0.0])) @ inv.T      # direction from depth 1 to depth 0
    tmax = np.linalg.norm(d[:3])
    d3 = d[:3] / tmax
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o[:, :3], 0.0, d3, tmax
    with capi.Context(64, 48) as ctx:
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.actualize_image("Shadow Map", D32, S, S)
        smap = _render(ctx, _pfd(sc, pv), S)
        t, _, _ = ctx.trace_explicit(rays, any_hit=False)
    got = smap[py, px].astype(np.float64)
    hit = t >= 0
    z = 1.0 - t.astype(np.float64) / tmax
    both = hit & (got > 0)
    err = np.abs(z[both] - got[both])
    # the pass snaps vertices to 1/256 texel (up to sqrt(2)/512 texel of displacement): on a surface seen edge-on from the light that
    # moves the depth by the map's own slope over that distance, which is allowed on top of the 1e-5
    m = smap.astype(np.float64)
    qx, qy = px[both], py[both]
    slope = np.max([np.abs(m[qy, np.clip(qx + k, 0, S - 1)] - m[qy, qx]) for k in (-1, 1)]
                   + [np.abs(m[np.clip(qy + k, 0, S - 1), qx] - m[qy, qx]) for k in (-1, 1)], axis=0)
    close = err <= 1e-5 + 0.003 * slope
    print(f"[shadow map] BVH: {int(hit.sum())} hits of {n}, depth within 1e-5 on {np.mean(err <= 1e-5)*100:.4f}% and within 1e-5 + the snapping "
          f"allowance on {close.mean()*100:.4f}% of {int(both.sum())}")
    assert close.mean() >= 0.999
    osc = O.OracleScene(sc)
    bad = np.flatnonzero(hit != (got > 0))
    for i in bad[:64]:
        margin = osc.brute_force(rays[i, :3], rays[i, 4:7], 0.0, float(rays[i, 7]))[2]
        assert margin <= 5e-3, f"texel ({px[i]}, {py[i]}): hit {bool(hit[i])} but map {got[i]} and no edge nearby (margin {margin:.2e})"
    print(f"[shadow map] BVH: {len(bad)} hit / covered mismatches, {min(len(bad), 64)} classified as edge grazes")
    assert len(bad) <= 0.001 * n


def _pcf_shadow(pfd, depth, smap):
    """composition.frag's rasterised shadow term (SHADOW_BIAS_MATRIX * projview, 16 bilinear taps 1/4096 apart, bias 1e-4), in double."""
    H, W = depth.shape
    S = smap.shape[0]
    inv = np.asarray(pfd["camera_viewproj_inverse"], np.float64).reshape(4, 4).T
    pv = np.asarray(pfd["directional_light"]["projview"], np.float64).reshape(4, 4).T
    y, x = np.mgrid[0:H, 0:W]
    with np.errstate(all="ignore"):
        q = np.stack([(x + 0.5) / W * 2 - 1, (y + 0.5) / H * 2 - 1, depth.astype(np.float64), np.ones((H, W))], -1) @ inv.T
        lp = np.concatenate([q[..., :3] / q[..., 3:], np.ones((H, W, 1))], -1) @ pv.T
        sx, sy, sz = 0.5 * lp[..., 0] + 0.5, 0.5 * lp[..., 1] + 0.5, lp[..., 2]
        m, acc = smap.astype(np.float64), np.zeros((H, W))
        for i in range(16):
            u = (sx + (-1.5 + (i >> 2)) / 4096.0) * S - 0.5
            v = (sy + (-1.5 + (i & 3)) / 4096.0) * S - 0.5
            x0, y0 = np.nan_to_num(np.floor(u)).astype(np.int64), np.nan_to_num(np.floor(v)).astype(np.int64)
            a, b = u - x0, v - y0
            g = lambda yy, xx: m[np.mod(yy, S), np.mod(xx, S)]
            ds = (1 - a) * (1 - b) * g(y0, x0) + a * (1 - b) * g(y0, x0 + 1) + (1 - a) * b * g(y0 + 1, x0) + a * b * g(y0 + 1, x0 + 1)
            acc += ~(sz < ds - 1e-4)
    return acc / 16.0


def test_plausible_against_ray_traced_shadows():
    """Where the two shadow techniques can disagree: the shadow map's fixed 1e-4 depth bias with a +-1.5-texel PCF footprint darkens
    lit surfaces that slope away from the light (the taps on the light's side compare against nearer depths), and the ray-traced
    shadow jitters inside the sun's cone. Measured with the CPU oracle on this scene (fitted window, 4096^2, 160 x 120): the PCF term's
    majority (>= 8 of 16 taps lit) agrees with the ray-traced mask on 95.9 % of the geometry pixels; bar 94 %."""
    W, H = 160, 120
    sc = scenes.tiny_scene(width=W, height=H)
    pfd = _pfd(sc, _fitted(sc), W, H)
    with capi.Context(W, H) as ctx:
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        path = HP.HybridRenderPath(ctx, W, H, composition=T.VK_FORMAT_B8G8R8A8_SRGB)
        ctx.update_per_frame_ubo(pfd)
        g = path.gsets[0]
        ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
        ctx.gbuffer_pass(W, H)
        path.shadow_map_pass()
        ctx.set_option(capi.OPT_TRACE_AO, 0)
        ctx.set_option(capi.OPT_TRACE_REFLECTIONS, 0)
        path.raytrace_pass()
        depth, smap, rt = ctx.image_download(g[HP.N_DEPTH]), ctx.image_download(HP.N_SHADOW_MAP), ctx.image_download(HP.N_RT)
    sh = _pcf_shadow(pfd, depth, smap)
    geo = depth > 0
    agree = float(np.mean((sh[geo] >= 0.5) == (rt[..., 0].astype(np.float32)[geo] == 1)))
    print(f"[shadow map] shadow-map majority vs ray-traced mask: {agree*100:.2f}% of {int(geo.sum())} pixels")
    assert agree >= 0.94


def test_host_frame_with_rasterised_shadows_and_ssao():
    W, H = 256, 144
    sc = scenes.sponza_like(30_000, seed=8, width=W, height=H, n_clutter=30)
    pfd = _pfd(sc, _fitted(sc), W, H)
    osc = O.OracleScene(sc)
    with host_api.Renderer(W, H) as r:
        r.load_scene(sc)
        r.set_modes(shadow=host_api.SHADOW_MODE_RASTERIZED, ao=host_api.AO_MODE_SSAO, reflection=host_api.REFLECTION_MODE_OFF)
        r.set_gbuffer_producer(True)
        r.set_shadow_map_producer(True)
        assert "Shadow Map Pass" in r.execution_order()
        r.render(pfd)
        out = r.ctx.image_download(HP.N_RENDER_OUTPUT)
        smap = r.ctx.image_download(HP.N_SHADOW_MAP)
    g = osc.gbuffer(pfd, W, H)
    want_map = SM.shadow_map(sc, pfd, 4096, 4096)
    _assert_bits(smap, want_map, "host graph 4096^2")
    ssao = O.ssao_blur(pfd, O.ssao(pfd, g["depth"], g["normals"], 0.75))
    rt = np.ones((H, W, 2), np.float16)
    want = O.composition(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], rt, 1, 1, 2, ssao_img=ssao, shadow_map=want_map,
                         out_format=T.VK_FORMAT_B8G8R8A8_SRGB)
    code = np.abs(out.astype(np.int32) - want.astype(np.int32))
    print(f"[shadow map] host RENDER_OUTPUT: exact {np.mean(code == 0)*100:.3f}%, within one code {np.mean(code.max(-1) <= 1)*100:.3f}%")
    assert np.mean(code.max(-1) <= 1) >= 0.995


def test_partition_ranks_render_the_whole_map():
    W, H, world, S = 320, 64 * 2 + 17, 2, 512
    sc = scenes.sponza_like(20_000, seed=3, width=W, height=H, n_clutter=30)
    pfd = _pfd(sc, _fitted(sc), W, H)

    def make():
        ctx = capi.Context(W, H)
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        return ctx, HP.HybridRenderPath(ctx, W, H, rt_sets=2, ssao=True, composition=T.VK_FORMAT_B8G8R8A8_SRGB, shadow_map_size=(S, S))

    ref_ctx, ref_path = make()
    ranks = [make() for _ in range(world)]
    try:
        MG.setup_fused_partition_inprocess([c for c, _ in ranks], [p for _, p in ranks], motion_halo=24)
        ref_ctx.update_per_frame_ubo(pfd)
        ref_path.shadow_map_pass()
        want = ref_ctx.image_download(HP.N_SHADOW_MAP)
        assert np.array_equal(want, SM.shadow_map(sc, pfd, S, S))
        for r, (ctx, path) in enumerate(ranks):
            ctx.update_per_frame_ubo(pfd)
            path.shadow_map_pass()
            _assert_bits(ctx.image_download(HP.N_SHADOW_MAP), want, f"rank {r} of {world}")
    finally:
        for c, _ in ranks + [(ref_ctx, None)]:
            c.close()
