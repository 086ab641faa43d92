"""Shared helpers for the parity tests: synthetic inputs, error metrics, the C-ABI SVGF pass body."""
import functools

import numpy as np

from vulkanhybridrenderer_b200 import camera, scenes
from vulkanhybridrenderer_b200 import types as T

# Parity bar from BASELINE.json north_star: max abs 1e-3 on linear values, PSNR >= 60 dB vs the reference restatement.
MAX_ABS_TOL = 1e-3
PSNR_MIN_DB = 60.0


def psnr(a, b, peak=1.0):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    mse = np.mean((a - b) ** 2)
    return 200.0 if mse == 0 else 10.0 * np.log10(peak * peak / mse)


def compare(gpu, ref, what=""):
    g = np.asarray(gpu, np.float32); r = np.asarray(ref, np.float32)
    assert g.shape == r.shape, (g.shape, r.shape)
    both_nan = np.isnan(g) & np.isnan(r)
    d = np.where(both_nan, 0.0, np.abs(g - r))
    stats = dict(max_abs=float(np.nanmax(d)) if d.size else 0.0, psnr=psnr(np.nan_to_num(g), np.nan_to_num(r)),
                 exact=float(np.mean((g == r) | both_nan)) if d.size else 1.0, nan_mismatch=int(np.sum(np.isnan(g) != np.isnan(r))))
    return stats


def assert_parity(gpu, ref, what, max_abs=MAX_ABS_TOL, min_psnr=PSNR_MIN_DB, outlier_frac=0.0):
    """max-abs / PSNR bar of north_star. `outlier_frac` > 0 (SSAO only): that fraction of the values may exceed `max_abs` — the texture
    unit holds the filter coordinate with 8 fractional bits, so a depth tap is a step function of the sample position, and a last-bit
    difference between CUDA's sincosf and the C library's sinf / cosf moves about one sample in 10^5 across a 1/256 step; next to a depth
    edge that one tap shifts the pixel's occlusion by a few 1e-3."""
    s = compare(gpu, ref, what)
    print(f"[parity] {what}: max_abs={s['max_abs']:.3e} psnr={s['psnr']:.1f}dB exact={s['exact']*100:.3f}% nan_mismatch={s['nan_mismatch']}")
    assert s["nan_mismatch"] == 0, (what, s)
    if outlier_frac > 0.0 and s["max_abs"] > max_abs:
        d = np.abs(np.asarray(gpu, np.float32) - np.asarray(ref, np.float32))
        frac = float(np.mean(np.nan_to_num(d) > max_abs))
        print(f"[parity] {what}: {frac*100:.4f}% of the values beyond {max_abs:g} (allowed {outlier_frac*100:.4f}%)")
        assert frac <= outlier_frac and s["max_abs"] <= 0.05, (what, s, frac)
        s["max_abs"] = max_abs
    assert s["psnr"] >= min_psnr, (what, s)
    return s


def oracle_bilinear_setup(u, n):
    """The oracle's bilinear_setup in numpy (float32 arrays): the filter coordinate t = fl(fl(u n) - 0.5) snapped to 1/256 as
    floor(t 256 + 0.5) / 256; returns (texel floor, unwrapped, as int64; weight; t)."""
    f32 = np.float32
    uu = ((u * f32(n)).astype(f32) - f32(0.5)).astype(f32)
    s = (np.floor(((uu * f32(256)).astype(f32) + f32(0.5)).astype(f32)) * f32(0.00390625)).astype(f32)
    fl = np.floor(s)
    return fl.astype(np.int64), (s - fl).astype(f32), uu


@functools.lru_cache(maxsize=8)
def scene_and_gbuffer(width, height, tris=20000, seed=3, moving=False):
    """Scene + oracle G-buffers of two consecutive frames (CPU primary rays; test scaffolding)."""
    import checker as O
    sc = scenes.sponza_like(tris, seed=seed, width=width, height=height, n_clutter=40)
    osc = O.OracleScene(sc)
    seq = camera.FrameSequencer(width, height, sc.light)
    frames = []
    cam = sc.camera
    for f in range(3):
        if moving and f > 0:
            pos = cam.position + np.array([0.05, 0.0, 0.01])
            cam.set_pose(pos, cam.yaw + 0.002, cam.pitch)
        pfd = seq.next(cam)
        frames.append((pfd, osc.gbuffer(pfd, width, height)))
    return sc, osc, frames


CAMERA_CASES = ("default", "jitter", "finite_far", "far_origin")


@functools.lru_cache(maxsize=16)
def camera_case(name, width, height):
    """(scene, oracle scene, pfd, oracle G-buffer) of one camera of the screen-space parity tests:
      default     the second frame of scene_and_gbuffer: infinite reverse-Z, whose inverse has only m00, m11, m23, m32 and m33 set;
      jitter      a TAA-style sub-pixel offset in perspective[0, 2] and [1, 2]: the inverse is not sparse;
      finite_far  reverse-Z with a far plane at 60: the inverse's m33 is not zero, so the sky (depth 0) unprojects with w != 0;
      far_origin  scene and camera translated by ~10^3 (Primitive.transform and the camera pose): coordinates lose ten bits;
      mirrored    perspective[0, 0] negated (a horizontally mirrored image);
      narrow_fov  a 5e-5 rad vertical field of view: |camera_proj_inverse m00|, |m11| < 2^-14."""
    if name == "default":
        sc, osc, frames = scene_and_gbuffer(width, height)
        return (sc, osc) + frames[1]
    import checker as O
    sc = scenes.sponza_like(20000, seed=3, width=width, height=height, n_clutter=40)
    cam = sc.camera
    if name == "jitter":
        cam.perspective = cam.perspective.copy()
        cam.perspective[0, 2], cam.perspective[1, 2] = 0.37 * 2.0 / width, -0.61 * 2.0 / height
    elif name == "finite_far":
        zn, zf = np.float32(cam.znear), np.float32(60.0)
        cam.perspective = cam.perspective.copy()
        cam.perspective[2, 2], cam.perspective[2, 3] = zn / (zf - zn), zn * zf / (zf - zn)
    elif name == "far_origin":
        off = np.array([1000.3, 250.7, -700.1])
        sc.primitives = sc.primitives.copy()
        sc.primitives["transform"][:, 3, :3] += off.astype(np.float32)
        cam.set_pose(cam.position + off, cam.yaw, cam.pitch)
    elif name == "mirrored":
        cam.perspective = cam.perspective.copy()
        cam.perspective[0, 0] = -cam.perspective[0, 0]
    elif name == "narrow_fov":
        cam.perspective = camera.infinite_reverse_depth_projection(5e-5, width / height, cam.znear)
    else:
        raise ValueError(name)
    osc = O.OracleScene(sc)
    seq = camera.FrameSequencer(width, height, sc.light)
    seq.next(cam)
    pfd = seq.next(cam)
    return sc, osc, pfd, osc.gbuffer(pfd, width, height)


def ssao_sample_angles(pfd, xs, ys):
    """The 16 sample angles of SSAO pixels (xs, ys), [n, 16] float32: ssao.comp's seed_thread / random01 sequence (common.glsl:47-68;
    the angle is fl(fl(r 2) PI) = fl(r (2 PI)), the distance draws the next number)."""
    u32 = np.uint32
    s = ((np.asarray(ys, np.uint64) * int(pfd["display_size"][1]) + np.asarray(xs, np.uint64)) * int(pfd["frame_index"])).astype(np.uint64)
    s = (s & 0xFFFFFFFF).astype(u32)
    with np.errstate(over="ignore"):
        s = (s ^ u32(61)) ^ (s >> u32(16))
        s = s * u32(9)
        s = s ^ (s >> u32(4))
        s = s * u32(0x27d4eb2d)
        s = s ^ (s >> u32(15))
        angles = []
        for _ in range(16):
            for k in range(2):
                s = s ^ (s << u32(13)); s = s ^ (s >> u32(17)); s = s ^ (s << u32(5))
                if k == 0:
                    r = (u32(0x3f800000) | (s >> u32(9))).view(np.float32) - np.float32(1.0)
                    angles.append((r * np.float32(2.0 * float(np.float32(np.pi)))).astype(np.float32))
    return np.stack(angles, axis=-1)


def noise_integrated(H, W, seed):
    """(shadow, ao, var_s, var_ao) noise image: worst case for the edge-stopping weights (SURVEY §8d config 1)."""
    rng = np.random.default_rng(seed)
    a = np.empty((H, W, 4), np.float32)
    a[..., 0] = rng.integers(0, 2, (H, W))
    a[..., 1] = rng.integers(0, 3, (H, W)) * 0.5
    a[..., 2] = rng.uniform(0, 0.25, (H, W)) * (rng.uniform(size=(H, W)) > 0.3)
    a[..., 3] = rng.uniform(0, 0.25, (H, W))
    return a.astype(np.float16)


GBUF_IMAGES = {
    "Albedo": T.VK_FORMAT_B8G8R8A8_UNORM,
    "World Space Normals and Object IDs": T.VK_FORMAT_R16G16B16A16_SFLOAT,
    "Motion Vectors and Metallic Roughness": T.VK_FORMAT_R16G16B16A16_SFLOAT,
    "Depth": T.VK_FORMAT_D32_SFLOAT,
}
N_NORMALS = "World Space Normals and Object IDs"
N_MOTION = "Motion Vectors and Metallic Roughness"
N_DEPTH = "Depth"
N_RT = "Raytraced Shadows and Ambient Occlusion"
N_REFL = "Raytraced Reflections"
N_DENOISED = "Denoised Raytraced Shadows and Ambient Occlusion"
N_SSAO_RAW = "Screen Space Ambient Occlusion Raw"
N_SSAO = "Screen Space Ambient Occlusion"


class SvgfPassCABI:
    """The SVGF Denoise Pass body of hybrid_render_path.cpp:245-331 issued call by call through the C-ABI."""

    def __init__(self, ctx, W, H):
        self.ctx, self.W, self.H = ctx, W, H
        F4, F2 = T.VK_FORMAT_R16G16B16A16_SFLOAT, T.VK_FORMAT_R16G16_SFLOAT
        for name, fmt in ((N_NORMALS, F4), (N_MOTION, F4), (N_DEPTH, T.VK_FORMAT_D32_SFLOAT), (N_RT, F2), (N_DENOISED, F4)):
            ctx.actualize_image(name, fmt)
        pc = np.zeros((), T.SVGFPushConstants)
        pc["integrated_shadow_and_ao"] = (ctx.upload_new_storage_image(W, H, F4), ctx.upload_new_storage_image(W, H, F4))
        pc["prev_frame_normals_and_object_ids"] = ctx.upload_new_storage_image(W, H, F4)
        pc["shadow_and_ao_history"] = ctx.upload_new_storage_image(W, H, F4)
        pc["shadow_and_ao_moments_history"] = ctx.upload_new_storage_image(W, H, F2)
        self.pc = pc

    def run(self, want_iters=False):
        ctx, pc = self.ctx, self.pc
        gx, gy = self.W // 8 + (self.W % 8 != 0), self.H // 8 + (self.H % 8 != 0)
        ctx.bind_pass_images([N_NORMALS, N_MOTION, N_DEPTH, N_RT, N_DENOISED])
        ctx.dispatch("hybrid_render_path/svgf.comp", gx, gy, 1, pc)
        temporal = ctx.storage_image_download(int(pc["integrated_shadow_and_ao"][0])) if want_iters else None
        iters = []
        for i in range(5):
            pc["atrous_step"] = 1 << i
            ctx.dispatch("hybrid_render_path/svgf_atrous_filter.comp", gx, gy, 1, pc)
            if want_iters:
                iters.append(ctx.storage_image_download(int(pc["integrated_shadow_and_ao"][1])))
            if i == 0:
                ctx.blit_storage_to_storage(int(pc["integrated_shadow_and_ao"][1]), int(pc["shadow_and_ao_history"]))
            pc["integrated_shadow_and_ao"] = pc["integrated_shadow_and_ao"][::-1].copy()
        ctx.blit_transient_to_storage(N_NORMALS, int(pc["prev_frame_normals_and_object_ids"]))
        ctx.blit_storage_to_transient(int(pc["integrated_shadow_and_ao"][1]), N_DENOISED)
        pc["integrated_shadow_and_ao"] = pc["integrated_shadow_and_ao"][::-1].copy()
        return ctx.image_download(N_DENOISED), (np.stack(iters) if want_iters else None), temporal


def world_triangles(sc):
    """World-space triangle soup (float32, same evaluation order as the builders): (n, 3, 3) array."""
    out = []
    for p in sc.primitives:
        m = p["transform"].astype(np.float32)          # m[c][r]
        idx = sc.indices[int(p["index_offset"]): int(p["index_offset"]) + int(p["index_count"])].astype(np.int64) + int(p["vertex_offset"])
        pos = sc.vertices["pos"][idx].astype(np.float32)
        w = np.empty_like(pos)
        for r in range(3):
            w[:, r] = ((m[0, r] * pos[:, 0] + m[1, r] * pos[:, 1]) + m[2, r] * pos[:, 2]) + m[3, r]
        out.append(w.reshape(-1, 3, 3))
    return np.concatenate(out) if out else np.zeros((0, 3, 3), np.float32)


def brute_force_hits(tris, o, d, tmin, tmax):
    """Exact-ish (float64 Moller-Trumbore) test of one ray against every triangle.
    Returns (any_hit, closest_t, edge_margin) where edge_margin is the smallest normalised barycentric distance to an
    edge or to the [tmin, tmax] interval among triangles whose plane the ray crosses nearby — small values mean the
    ray grazes an edge / the interval end (an epsilon case)."""
    t64 = tris.astype(np.float64)
    o = np.asarray(o, np.float64); d = np.asarray(d, np.float64)
    e1 = t64[:, 1] - t64[:, 0]; e2 = t64[:, 2] - t64[:, 0]
    pv = np.cross(d[None, :], e2)
    det = np.einsum("ij,ij->i", e1, pv)
    ok = np.abs(det) > 0
    inv = np.where(ok, 1.0 / np.where(ok, det, 1.0), 0.0)
    tv = o[None, :] - t64[:, 0]
    u = np.einsum("ij,ij->i", tv, pv) * inv
    qv = np.cross(tv, e1)
    v = np.einsum("j,ij->i", d, qv) * inv
    t = np.einsum("ij,ij->i", e2, qv) * inv
    w = 1.0 - u - v
    inside = ok & (u >= 0) & (v >= 0) & (w >= 0) & (t > tmin) & (t < tmax)
    # margin: how far the nearest candidate is from flipping its classification
    bary_margin = np.minimum(np.minimum(np.abs(u), np.abs(v)), np.abs(w))
    t_margin = np.minimum(np.abs(t - tmin), np.abs(t - tmax)) / np.maximum(1.0, np.abs(t))
    near = ok & (u > -1e-3) & (v > -1e-3) & (w > -1e-3) & (t > tmin - 1e-3) & (t < tmax + 1e-3)
    margin = float(np.min(np.minimum(bary_margin, t_margin)[near])) if near.any() else 1.0
    return bool(inside.any()), (float(t[inside].min()) if inside.any() else -1.0), margin


def classify_mask_mismatches(osc, pfd, depth, normals, gpu_sa, ref_sa, ao_spp, what, flags=3, max_margin=1e-4, max_checked=64):
    """north_star: visibility-mask mismatches must be "confined to self-intersection-epsilon / grazing cases". Every pixel on which the GPU's
    shadow / AO texel differs from the checker's is re-traced here: the pixel's rays are regenerated (oracle, same statements as raygen.rgen) and
    each one is tested against EVERY triangle in double precision; a mismatching pixel must own at least one ray whose nearest candidate lies
    within `max_margin` of flipping (barycentric distance to an edge, or relative distance of t to tMin / tMax). Returns the number classified."""
    import oracle_lib as OL
    bad = np.argwhere(np.any(np.asarray(gpu_sa).view(np.uint16) != np.asarray(ref_sa).view(np.uint16), axis=-1))
    worst = 0.0
    for y, x in bad[:max_checked]:
        rays = OL.raygen_pixel_rays(pfd, depth, normals, x, y, ao_spp)
        use = [i for i in range(len(rays)) if (i == 0 and flags & 1) or (i > 0 and flags & 2)]
        margins = [osc.brute_force(rays[i, :3], rays[i, 4:7], rays[i, 3], rays[i, 7])[2] for i in use]
        assert margins, (what, x, y)
        m = min(margins)
        worst = max(worst, m)
        assert m <= max_margin, f"{what}: pixel ({x}, {y}) differs but none of its rays grazes anything (smallest margin {m:.3e}): a real miss, not an epsilon case"
    print(f"[masks] {what}: {len(bad)} mismatching pixels of {gpu_sa.shape[0] * gpu_sa.shape[1]}, {min(len(bad), max_checked)} re-traced by brute force, "
          f"all grazing (largest margin {worst:.2e})")
    return len(bad)
