"""The "Shadow Map Pass" specification on the CPU: oracle/oracle_shadow_map.cpp (vo_shadow_map) against an independent
double-precision evaluation, its fill rule, guard-band clipping and special cases; camera.light_projview against the scene
loader; the C-ABI entry point on a validation-only context."""
import numpy as np
import pytest

import helpers as Hh
import shadow_map_lib as SM
from vulkanhybridrenderer_b200 import camera, capi, gltf_export, host_api, scenes
from vulkanhybridrenderer_b200 import types as T


class _Soup:
    """A scene of explicit world-space triangles: one primitive, identity transform."""

    def __init__(self, tris):
        tris = np.asarray(tris, np.float32).reshape(-1, 3, 3)
        self.vertices = np.zeros(3 * len(tris), T.Vertex)
        self.vertices["pos"] = tris.reshape(-1, 3)
        self.indices = np.arange(3 * len(tris), dtype=np.uint32)
        self.primitives = np.zeros(1, T.Primitive)
        self.primitives["transform"] = np.eye(4, dtype=np.float32)
        self.primitives["index_count"] = 3 * len(tris)


def _pfd(projview):
    pfd = np.zeros((), T.PerFrameData)
    pfd["directional_light"]["projview"] = np.asarray(projview, np.float32).reshape(4, 4)
    return pfd


def _texel_projview(W, H):
    """World (x, y) -> map coordinates (x, y) exactly (texel centres at k + 0.5), z -> depth."""
    m = np.array([[2.0 / W, 0, 0, -1], [0, 2.0 / H, 0, -1], [0, 0, 1, 0], [0, 0, 0, 1]])
    return camera.to_glm(m)


def _reference_map(tris, pv, W, H, tie_margin=1e-3):
    """Double-precision depth of the first surface (largest depth in [0, 1]) through every texel centre, over the triangles as the
    pass sees them: projected in fp32 in the pass's order and snapped to 1/256 texel (DESIGN §2). Returns (depth, tie) where `tie`
    marks texels whose centre lies within `tie_margin` texel of a projected edge of a triangle that reaches it."""
    m = np.asarray(pv, np.float32).reshape(4, 4)      # m[c, r]
    t = np.asarray(tris, np.float32)
    one = np.float32(1.0)
    clip = [((m[0, r] * t[..., 0] + m[1, r] * t[..., 1]) + (m[2, r] * t[..., 2] + m[3, r] * one)) for r in range(3)]
    hw, hh = np.float32(0.5) * np.float32(W), np.float32(0.5) * np.float32(H)
    X = np.rint((hw * clip[0] + hw).astype(np.float64) * 256.0) / 256.0
    Y = np.rint((hh * clip[1] + hh).astype(np.float64) * 256.0) / 256.0
    Z = clip[2].astype(np.float64)
    depth = np.zeros((H, W))
    tie = np.zeros((H, W), bool)
    for k in range(len(t)):
        x, y, z = X[k], Y[k], Z[k]
        area = (x[1] - x[0]) * (y[2] - y[0]) - (y[1] - y[0]) * (x[2] - x[0])
        if area == 0 or (z < 0).all() or (z > 1).all():
            continue
        px0, px1 = max(0, int(np.floor(x.min() - 0.5)) - 1), min(W - 1, int(np.ceil(x.max() - 0.5)) + 1)
        py0, py1 = max(0, int(np.floor(y.min() - 0.5)) - 1), min(H - 1, int(np.ceil(y.max() - 0.5)) + 1)
        if px0 > px1 or py0 > py1:
            continue
        sy, sx = np.mgrid[py0:py1 + 1, px0:px1 + 1] + 0.5
        s = np.sign(area)
        e, dist = [], []
        for a, b in ((1, 2), (2, 0), (0, 1)):
            ev = s * ((x[b] - x[a]) * (sy - y[a]) - (y[b] - y[a]) * (sx - x[a]))
            e.append(ev)
            dist.append(ev / np.hypot(x[b] - x[a], y[b] - y[a]))
        dmin = np.minimum(np.minimum(dist[0], dist[1]), dist[2])
        b1, b2 = e[1] / abs(area), e[2] / abs(area)
        zz = z[0] + b1 * (z[1] - z[0]) + b2 * (z[2] - z[0])
        inside = dmin > tie_margin
        near = (np.abs(dmin) <= tie_margin) & (zz >= -1e-6) & (zz <= 1 + 1e-6)
        tie[py0:py1 + 1, px0:px1 + 1] |= near | (inside & ((np.abs(zz) <= 1e-6) | (np.abs(zz - 1) <= 1e-6)))
        keep = inside & (zz >= 0) & (zz <= 1)
        blk = depth[py0:py1 + 1, px0:px1 + 1]
        blk[keep] = np.maximum(blk[keep], zz[keep])
    return depth, tie


def _scene_box(sc):
    p = Hh.world_triangles(sc).reshape(-1, 3)
    return p.min(0), p.max(0)


@pytest.mark.parametrize("window", ["reference", "fitted"])
def test_oracle_matches_double_precision_depth(window):
    W = H = 256
    sc = scenes.tiny_scene()
    d = sc.light["direction"][:3]
    pv = camera.light_projview(d) if window == "reference" else camera.fit_light_projview(d, *_scene_box(sc))
    got = SM.shadow_map(sc, _pfd(pv), W, H)
    want, tie = _reference_map(Hh.world_triangles(sc), pv, W, H)
    err = np.abs(got.astype(np.float64) - want)
    print(f"[shadow map] {window}: {int(np.sum(want > 0))} covered texels, {int(tie.sum())} edge / depth-range ties classified, "
          f"max |d| off ties {err[~tie].max():.2e}")
    assert err[~tie].max() <= 1e-6
    assert tie.mean() < 0.02
    assert np.sum(want[~tie] > 0) > 0.1 * W * H          # the map actually sees the scene (the reference window clips half of it)


def test_fill_rule_tessellated_square_has_no_gaps():
    W = H = 32
    n = 12                                                   # vertices on texel centres 4.5 .. 16.5
    rng = np.random.default_rng(1)
    tris = []
    for j in range(n):
        for i in range(n):
            a, b, c, d = [(4.5 + i + di, 4.5 + j + dj, 0.5) for di, dj in ((0, 0), (1, 0), (0, 1), (1, 1))]
            quad = [(a, b, d), (a, d, c)] if rng.integers(2) else [(a, b, c), (b, d, c)]
            for tri in quad:                                 # both windings
                tris.append(tri if rng.integers(2) else tri[::-1])
    got = SM.shadow_map(_Soup(tris), _pfd(_texel_projview(W, H)), W, H)
    covered = got > 0
    want = np.zeros((H, W), bool)
    want[4:4 + n, 4:4 + n] = True                            # top and left boundaries in, right and bottom out
    assert np.array_equal(covered, want)
    assert np.all(got[covered] == np.float32(0.5))


@pytest.mark.parametrize("reverse", [False, True])
def test_fill_rule_lone_triangles(reverse):
    W = H = 16
    upper = [(2.5, 2.5, 0.25), (10.5, 2.5, 0.25), (2.5, 10.5, 0.25)]     # top edge, left edge, hypotenuse right / bottom
    lower = [(10.5, 10.5, 0.75), (2.5, 10.5, 0.75), (10.5, 2.5, 0.75)]   # bottom edge, right edge, hypotenuse top-left
    py, px = np.mgrid[0:H, 0:W]
    for tri, want in ((upper, (px >= 2) & (py >= 2) & (px + py < 12)), (lower, (px <= 9) & (py <= 9) & (px + py >= 12))):
        got = SM.shadow_map(_Soup([tri[::-1] if reverse else tri]), _pfd(_texel_projview(W, H)), W, H)
        assert np.array_equal(got > 0, want)


def test_triangle_crossing_the_guard_band():
    W = H = 32
    big = 2.0 ** 22                                           # beyond the 2^20-texel guard band on both axes
    z = np.float32([0.25, 0.25 + big * 1e-7, 0.25 + big * 2e-7])
    tri = [(8.0, 8.0, z[0]), (8.0 + big, 8.0, z[1]), (8.0, 8.0 + big, z[2])]
    got = SM.shadow_map(_Soup([tri]), _pfd(_texel_projview(W, H)), W, H)
    py, px = np.mgrid[0:H, 0:W] + 0.5
    want = z[0] + (px - 8.0) / big * (float(z[1]) - z[0]) + (py - 8.0) / big * (float(z[2]) - z[0])
    inside = (px > 8) & (py > 8)
    assert np.array_equal(got > 0, inside)
    assert np.abs(got[inside] - want[inside]).max() <= 1e-6


def test_zero_projview_clears_and_non_affine_is_rejected():
    sc = scenes.tiny_scene()
    assert not SM.shadow_map(sc, _pfd(np.zeros(16)), 64, 64).any()
    pv = camera.light_projview(sc.light["direction"][:3]).copy()
    pv[2, 3] = 0.5                                            # m[11]: a perspective term in the last row
    with pytest.raises(ValueError):
        SM.shadow_map(sc, _pfd(pv), 64, 64)
    pv = camera.light_projview(sc.light["direction"][:3]).copy()
    pv[0, 0] = np.nan
    with pytest.raises(ValueError):
        SM.shadow_map(sc, _pfd(pv), 64, 64)


def test_negative_zero_is_never_stored():
    W = H = 16
    mz = np.float32(-0.0)
    pv = _texel_projview(W, H)
    pv[0, 2] = pv[1, 2] = pv[3, 2] = mz                       # depth = (-0 x + -0 y) + (1 z + -0) = -0 for z = -0
    got = SM.shadow_map(_Soup([[(1, 1, mz), (14, 1, mz), (1, 14, mz)]]), _pfd(pv), W, H)
    assert not np.any(got.view(np.uint32) == 0x80000000)


@pytest.mark.parametrize("direction", [(-0.3, -1.0, 0.2), (0.5, -0.7, -0.4)])
def test_light_projview_matches_scene_loader(tmp_path, direction):
    sc = scenes.sponza_like(2000, seed=5, width=64, height=48, n_clutter=5)
    sc.light = camera.directional_light(direction)
    got = host_api.parse_gltf(gltf_export.export(sc, tmp_path / "light.glb"))["light"]
    assert np.abs(camera.light_projview(got["direction"]) - got["projview"]).max() <= 1e-6


def test_pass_needs_a_device():
    with capi.Context(64, 48, device=host_api.DEVICE_NONE) as ctx:
        ctx.actualize_image("Shadow Map", T.VK_FORMAT_D32_SFLOAT, 64, 64)
        ctx.bind_pass_images(["Shadow Map"])
        with pytest.raises(capi.VhrError) as e:
            ctx.shadow_map_pass()
        assert "status -2" in str(e.value) and "VHR_DEVICE_NONE" in str(e.value)
