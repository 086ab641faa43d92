"""GPU: the shading after a ray hit and the texture unit, bit for bit against the CPU oracle on IDENTICAL hits.

The frame-level tests compare the GPU with the oracle through each side's own traversal: the GPU finds its hits in fp32 and the oracle in
double, so the two sides shade slightly different points and those tests carry tolerances. Here vhr_debug_shade_hits and vo_shade_hits
run the per-hit code of the passes (the same functions the production kernels and the oracle's frame loops call) on the same
(geometry, primitive, barycentrics) records, so there is no reason for any tolerance: every comparison is on the bits (fp32 as uint32,
fp16 as uint16, packed words as words).

Two cases create a NaN on purpose, and only there are NaNs compared as a class (DESIGN.md section 2):
  * the texture unit's LINEAR filter at a non-finite filter coordinate (a coordinate that is NaN or infinite, or so large that
    (s n - 0.5) 256 overflows): the weights are NaN, so all four channels are NaN on both sides;
  * the G-buffer normal of a normal-mapped hit whose tangent, made orthogonal to the normal, is exactly zero (the tangent of the
    degenerate-frame primitive is parallel to its normal): normalize(0) is NaN in the shaders' arithmetic, and the fp16 store keeps
    a NaN, whose payload the two sides encode differently.
"""
import numpy as np
import pytest

import oracle_lib as O
from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu

f32 = np.float32
NEAREST, LINEAR = 0, 1
REPEAT, MIRROR, CLAMP, BORDER = 0, 1, 2, 3
UNORM, SRGB = T.VK_FORMAT_R8G8B8A8_UNORM, T.VK_FORMAT_R8G8B8A8_SRGB
W, H = 320, 180


def _records(g, pid, u, v, x=0, y=0):
    n = len(np.atleast_1d(g))
    r = np.zeros(n, T.ShadeRecord)
    r["g"], r["pid"], r["u"], r["v"], r["x"], r["y"] = g, pid, np.asarray(u, f32), np.asarray(v, f32), x, y
    return r


def _same_bits(got, want, what):
    """Word-for-word equality of two [n, words] uint32 arrays."""
    rows = np.nonzero((got != want).any(axis=1))[0]
    assert len(rows) == 0, f"{what}: {len(rows)} of {len(got)} records differ; first {rows[:8].tolist()}: gpu {got[rows[:3]].tolist()} oracle {want[rows[:3]].tolist()}"


def _is_nan32(w):
    return ((w & 0x7f800000) == 0x7f800000) & ((w & 0x007fffff) != 0)


def _is_nan16(h):
    return ((h & 0x7c00) == 0x7c00) & ((h & 0x03ff) != 0)


# ---- the texture unit ---------------------------------------------------------------------------------------------------------------
def _axis_coords(n, rng):
    """Texture coordinates along one axis of an n-texel image, where a sampler's arithmetic goes wrong."""
    nf = f32(n)
    i = np.arange(n) if n <= 48 else np.unique(np.concatenate([np.arange(4), n - 1 - np.arange(4), rng.integers(0, n, 24)]))
    centres = ((i + 0.5) / n).astype(f32)
    edges = (np.concatenate([i, [n]]) / n).astype(f32)
    base = np.concatenate([centres, edges])
    near = np.concatenate([base, np.nextafter(base, f32(np.inf)), np.nextafter(base, f32(-np.inf))])
    # LINEAR tie points: fl(s n - 0.5) 256 + 0.5 is an integer, i.e. the sub-texel rounding of the filter coordinate is a tie
    m = rng.integers(-2 * 256 * n, 3 * 256 * n, 64)
    s = ((m + 0.5) / 256.0 + 0.5) / n
    s = np.concatenate([s.astype(f32), np.nextafter(s.astype(f32), f32(np.inf)), np.nextafter(s.astype(f32), f32(-np.inf))])
    with np.errstate(all="ignore"):
        t = (s * nf - f32(0.5)) * f32(256.0) + f32(0.5)
    ties = s[t == np.floor(t)]
    assert len(ties) >= 8
    # signed zeros, whole numbers, one and two periods outside the image (MIRRORED_REPEAT: the period is 2n texels = 2 in s)
    periods = np.concatenate([centres[:6] + k for k in (-4, -2, -1, 1, 2, 3)]).astype(f32)
    special = np.array([0.0, -0.0, 1.0, -1.0, 2.0, -2.0], f32)
    # |s n| crossing 2^14 (the fast path of the screen-space bilinear setup), 2^23 / 2^24 (fp32 loses the fraction / odd integers)
    # and 1e9 (the guard on the texel index)
    big = np.array([2.0 ** 14, 2.0 ** 23, 2.0 ** 24, 1e9, 1e9 * 256.0], np.float64) / n
    big = big.astype(f32)
    big = np.concatenate([big, np.nextafter(big, f32(np.inf)), np.nextafter(big, f32(-np.inf))])
    big = np.concatenate([big, -big])
    extreme = np.array([np.finfo(f32).max, -np.finfo(f32).max, np.inf, -np.inf, np.nan, 1e-40, -1e-40, 1.4e-45, np.finfo(f32).tiny], f32)
    bits = rng.integers(0, 2 ** 32, 24, dtype=np.uint64).astype(np.uint32).view(f32)
    return np.concatenate([near, ties, periods, special, big, extreme, bits]).astype(f32)


def _texture_bank(rng):
    """Every format x mag filter x address-mode pair at sizes 1x1 ... 256x256, plus one texture wider than 2^14 texels. The min filter
    is always the other filter: a sampler that applied it would show."""
    sizes = [(1, 1), (1, 5), (7, 1), (3, 3), (61, 37), (256, 256)]
    bank = []
    for fmt in (UNORM, SRGB):
        for mag in (NEAREST, LINEAR):
            for wu in range(4):
                for wv in range(4):
                    for (w, h) in sizes:
                        bank.append((w, h, fmt, (mag, 1 - mag, wu, wv)))
    for fmt, mag, wu in ((UNORM, LINEAR, REPEAT), (SRGB, NEAREST, MIRROR), (SRGB, LINEAR, BORDER)):
        bank.append((20_000, 1, fmt, (mag, 1 - mag, wu, CLAMP)))
    out = []
    for w, h, fmt, smp in bank:
        rgba = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        rgba.reshape(-1, 4)[0, 3] = 0                       # alpha 0 and 255 present in every texture
        rgba.reshape(-1, 4)[-1, 3] = 255
        out.append((rgba, fmt, smp))
    return out


def test_texture_unit_bit_exact_on_every_sampler_configuration():
    rng = np.random.default_rng(20261022)
    bank = _texture_bank(rng)
    osc = O.OracleScene(scenes.Scene(np.zeros(0, T.Vertex), np.zeros(0, np.uint32), np.zeros(0, T.Primitive), None, None, "textures"))
    recs, lin, nan_expected, border = [], [], [], []
    with capi.Context(64, 64) as ctx:
        ctx.update_per_frame_ubo(np.zeros((), T.PerFrameData))
        for k, (rgba, fmt, smp) in enumerate(bank):
            h, w = rgba.shape[:2]
            assert ctx.upload_texture_from_data(rgba, fmt, smp) == k
            assert osc.add_texture(rgba, fmt, smp) == k
            su, sv = _axis_coords(w, rng), _axis_coords(h, rng)
            # every u against a few v and every v against a few u, plus random pairs
            s = np.concatenate([su, np.repeat(f32(0.5 / h), len(sv)), rng.choice(su, 96)])
            t = np.concatenate([np.repeat(f32(0.5 / w) if h > 1 else f32(0.25), len(su)), sv, rng.choice(sv, 96)])
            s = np.concatenate([s, rng.choice(su, 32)]); t = np.concatenate([t, rng.choice(sv, 32)])
            s, t = s.astype(f32), t.astype(f32)
            recs.append(_records(np.full(len(s), k), 0, s, t))
            with np.errstate(all="ignore"):
                fin = np.isfinite((s * f32(w) - f32(0.5)) * f32(256.0)) & np.isfinite((t * f32(h) - f32(0.5)) * f32(256.0))
                outside = lambda c, m: ~((c >= 0) & (c < 1)) if m == BORDER else np.zeros(len(c), bool)
            lin.append(np.full(len(s), smp[0] == LINEAR))
            nan_expected.append((smp[0] == LINEAR) & ~fin)
            border.append(outside(s, smp[2]) | outside(t, smp[3]))
        rec = np.concatenate(recs)
        got = ctx.shade_hits(T.SHADE_TEXTURE, rec)
    want = osc.shade_hits(np.zeros((), T.PerFrameData), T.SHADE_TEXTURE, rec)
    nan_expected, lin, border = np.concatenate(nan_expected), np.concatenate(lin), np.concatenate(border)
    # the documented NaN case: a LINEAR lookup at a non-finite filter coordinate gives NaN in all four channels on both sides
    assert (_is_nan32(got[:, :4]).all(axis=1) == nan_expected).all() and (_is_nan32(want[:, :4]).all(axis=1) == nan_expected).all()
    assert not _is_nan32(got[~nan_expected, :4]).any()
    _same_bits(got[~nan_expected], want[~nan_expected], "texture(textures[i], uv)")
    assert (got[:, 4:] == 0).all()
    opaque_black = np.array([0, 0, 0, 0x3f800000], np.uint32)
    n_border_black = int((got[~lin, :4] == opaque_black).all(axis=1)[border[~lin]].sum())
    counts = dict(records=len(rec), textures=len(bank), linear=int(lin.sum()), nearest=int((~lin).sum()), nan_by_design=int(nan_expected.sum()),
                  border_coordinate=int(border.sum()), nearest_border_texel=n_border_black)
    print("\n[texture unit]", counts)
    assert counts["nan_by_design"] >= 500 and counts["border_coordinate"] >= 5000 and counts["nearest_border_texel"] >= 1000


# ---- hits -----------------------------------------------------------------------------------------------------------------------------
def _unit(v):
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(f32)


def _soup(rng, n_tris, uv_lo=-0.6, uv_hi=2.4):
    """n_tris separate triangles (3 vertices each) with random positions, unit normals, tangents and uv0 (tangent.w = +1)."""
    v = np.zeros(3 * n_tris, T.Vertex)
    v["pos"] = rng.uniform(-1.0, 1.0, (3 * n_tris, 3))
    v["normal"] = _unit(rng.normal(size=(3 * n_tris, 3)))
    v["tangent"][:, :3] = _unit(rng.normal(size=(3 * n_tris, 3)))
    v["tangent"][:, 3] = 1.0
    v["uv0"] = rng.uniform(uv_lo, uv_hi, (3 * n_tris, 2))
    v["uv1"] = v["uv0"]
    return v, np.arange(3 * n_tris, dtype=np.uint32)


def _transform(rot_yaw, rot_pitch, scale, translation):
    m = scenes._trs(translation, rot_yaw, scale, rot_pitch)
    return np.asarray(m, np.float32).T


def _material(p, color=(0.7, 0.6, 0.5, 1.0), tex=-1, mr=-1, nm=-1, metallic=0.5, roughness=0.5, alpha_mask=0, cutoff=0.5):
    m = p["material"]
    m["base_color"] = color
    m["base_color_texture"], m["metallic_roughness_texture"], m["normal_map"] = tex, mr, nm
    m["metallic_factor"], m["roughness_factor"] = metallic, roughness
    m["alpha_mask"], m["alpha_cutoff"] = alpha_mask, cutoff


ALPHA_K = 128          # the alpha-mask cutoff is exactly the decoded texel alpha ALPHA_K / 255


def _build_world():
    """The procedural textured hall plus hand-built primitives; returns (scene, {name: list of geometry indices})."""
    rng = np.random.default_rng(7)
    sc = scenes.add_procedural_textures(scenes.sponza_like(20_000, seed=3, width=W, height=H, n_clutter=30), size=32)
    n_hall = len(sc.primitives)
    # extra textures covering more sampler configurations (appended after the procedural bank: slots = list index)
    tex0 = len(sc.textures)
    extra = [((7, 5), SRGB, (NEAREST, LINEAR, MIRROR, BORDER)), ((16, 16), SRGB, (LINEAR, NEAREST, CLAMP, MIRROR)),
             ((1, 1), SRGB, (LINEAR, NEAREST, REPEAT, REPEAT)), ((9, 13), UNORM, (NEAREST, LINEAR, BORDER, CLAMP)),
             ((32, 8), UNORM, (LINEAR, NEAREST, MIRROR, REPEAT)), ((5, 5), UNORM, (LINEAR, NEAREST, BORDER, BORDER))]
    for (w, h), fmt, smp in extra:
        sc.textures.append(scenes.Texture(rng.integers(0, 256, (h, w, 4), dtype=np.uint8), fmt, smp))
    T_COL, T_COL2, T_ONE, T_MR, T_NM, T_NM2 = range(tex0, tex0 + 6)
    # the alpha texture: one texel per alpha value around the cutoff, sampled NEAREST at its centre
    alphas = np.array([ALPHA_K - 1, ALPHA_K, ALPHA_K + 1, 0, 255], np.uint8)
    at = np.zeros((1, len(alphas), 4), np.uint8)
    at[0, :, :3] = rng.integers(0, 256, (len(alphas), 3))
    at[0, :, 3] = alphas
    sc.textures.append(scenes.Texture(at, SRGB, (NEAREST, LINEAR, CLAMP, CLAMP)))
    T_ALPHA = tex0 + 6

    verts, inds, prims = [sc.vertices], [sc.indices], [sc.primitives]
    v_off, i_off = len(sc.vertices), len(sc.indices)
    groups = {}

    def add(name, v, ix, transform, **mat):
        nonlocal v_off, i_off
        p = np.zeros((), T.Primitive)
        p["transform"] = transform
        _material(p, **mat)
        p["vertex_offset"], p["index_offset"], p["index_count"] = v_off, i_off, len(ix)
        verts.append(v); inds.append(ix); prims.append(p.reshape(1))
        groups.setdefault(name, []).append(n_hall + sum(len(q) for q in prims[1:]) - 1)
        v_off += len(v); i_off += len(ix)

    ident = np.eye(4, dtype=np.float32)
    v, ix = _soup(rng, 24)
    add("mirrored", v, ix, _transform(0.7, 0.3, (-1.3, 0.8, 1.1), (2.0, 1.5, -3.0)), tex=T_COL, mr=T_MR, nm=T_NM, metallic=1.0, roughness=1.0)
    v, ix = _soup(rng, 24)
    v["tangent"][:, 3] = -1.0
    add("rot_scale_tangent_w_neg", v, ix, _transform(-1.1, 0.9, (0.3, 2.5, 1.7), (-4.0, 2.0, 1.0)), tex=T_COL2, mr=5, nm=T_NM2, metallic=0.8,
        roughness=0.9)
    v, ix = _soup(rng, 24)
    v["tangent"][:, 3] = np.where(np.arange(len(v)) % 2 == 0, 1.0, -1.0)     # the sign flips across each triangle
    add("rot_scale_tangent_w_mixed", v, ix, _transform(2.0, -0.4, (1.5, 0.5, 0.9), (0.0, 3.0, 0.0)), tex=T_ONE, nm=6)
    v, ix = _soup(rng, 24)
    v["normal"] = np.array([0.0, 0.0, 1.0], f32)
    v["tangent"][:, :3] = v["normal"]                                           # tangent parallel to the normal: a degenerate frame
    add("degenerate_frame", v, ix, ident, tex=T_COL, nm=T_NM)
    # alpha mask with the cutoff exactly at a decoded texel alpha: each triangle's uv0 is one texel centre of the alpha texture
    v, ix = _soup(rng, 5 * 4)
    v["uv0"][:, 0] = ((np.arange(len(v)) // 3 % len(alphas)) + 0.5) / len(alphas)
    v["uv0"][:, 1] = 0.5
    cutoff = f32(ALPHA_K) / f32(255.0)
    add("alpha_cutoff_tie", v, ix, ident, tex=T_ALPHA, alpha_mask=1, cutoff=cutoff)
    add("alpha_texel_no_mask", v, ix, ident, tex=T_ALPHA, alpha_mask=0, cutoff=cutoff)
    v, ix = _soup(rng, 8)
    add("alpha_zero_factor", v, ix, ident, color=(0.4, 0.5, 0.6, 0.0))
    add("alpha_cutoff_factor_tie", v, ix, ident, color=(0.4, 0.5, 0.6, float(cutoff)), alpha_mask=1, cutoff=cutoff)
    # metallic / roughness factors outside [0, 1], with and without a metallic-roughness texture
    v, ix = _soup(rng, 16)
    for k, (mt, rg) in enumerate(((-0.5, 1.7), (2.5, -0.3), (1.25, 0.01), (-2.0, 3.0))):
        add("mr_out_of_range", v, ix, _transform(0.1 * k, 0.0, (1, 1, 1), (0.5 * k, 0, 0)), tex=T_COL if k % 2 else -1, mr=T_MR if k < 2 else -1,
            metallic=mt, roughness=rg)
    # many small primitives so that geometry indices pass 2048 and 4096 (fp16 stores of (float)g round above 2048)
    v, ix = _soup(rng, 4)
    cycle = [dict(tex=T_COL, nm=T_NM, mr=T_MR), dict(), dict(tex=T_ALPHA, alpha_mask=1, cutoff=cutoff), dict(tex=2, nm=6),
             dict(color=(0.2, 0.9, 0.1, 0.0)), dict(tex=T_COL2, mr=4, metallic=1.5, roughness=-0.5)]
    n_many = 4400 - n_hall - sum(len(g) for g in groups.values())
    for k in range(n_many):
        add("many", v, ix, _transform(0.01 * k, 0.003 * k, (1.0 + (k % 3) * 0.5, 1.0, 0.7), (k % 17, (k // 17) % 5, -(k % 7))), **cycle[k % len(cycle)])
    sc.vertices, sc.indices, sc.primitives = np.concatenate(verts), np.concatenate(inds), np.concatenate(prims)
    assert len(sc.primitives) == 4400
    return sc, groups


BARY = [(0.0, 0.0), (1.0, 0.0), (0.0, 1.0), (1.0 / 3.0, 1.0 / 3.0), (0.5, 0.0), (0.0, 0.5), (0.5, 0.5)]


def _bary_set(rng, n):
    """The barycentric pairs every synthetic triangle is shaded at: corners, centroid, edge midpoints, u + v = 1 exactly and one ulp either
    side, random."""
    u = [f32(a) for a, _ in BARY]
    v = [f32(b) for _, b in BARY]
    for a in (f32(0.3), f32(0.7), f32(0.123456)):
        b = f32(1.0) - a
        u += [a, a, a]
        v += [b, np.nextafter(b, f32(2.0)), np.nextafter(b, f32(-1.0))]
    uv = np.array([u, v], f32).T
    r = rng.uniform(0.0, 1.0, (n, 2)).astype(f32)
    r = np.where(r.sum(1, keepdims=True) > 1.0, 1.0 - r, r).astype(f32)
    return np.concatenate([uv, r])


@pytest.fixture(scope="module")
def world():
    sc, groups = _build_world()
    rng = np.random.default_rng(11)
    cam = sc.camera
    seq = camera.FrameSequencer(W, H, sc.light)
    pfd0 = seq.next(cam)
    cam.set_pose(cam.position + np.array([0.3, 0.05, -0.2]), cam.yaw + 0.03, cam.pitch - 0.01)
    pfd1 = seq.next(cam)
    # the second set: a light that grazes the floor from below the horizon for part of the hits (negative N.L)
    pfd2 = pfd1.copy()
    pfd2["directional_light"] = camera.directional_light((0.6, 0.25, -0.4), color=(1.0, 0.8, 0.6), intensity=12.0)
    ctx = capi.Context(W, H)
    ctx.load_scene(sc)
    osc = O.OracleScene(sc)
    yield dict(sc=sc, groups=groups, ctx=ctx, osc=osc, pfds=[pfd1, pfd2], rng=rng)
    ctx.close()


def _synthetic_hits(world):
    sc, groups, rng = world["sc"], world["groups"], world["rng"]
    tri_counts = sc.primitives["index_count"] // 3
    special = sorted(g for name, gs in groups.items() if name != "many" for g in gs)
    many = groups["many"]
    hall = np.arange(len(sc.primitives) - len(special) - len(many))
    gs, ps = [], []
    for g in special + list(rng.choice(many, 400, replace=False)) + [many[-1], many[-2]]:
        for p in range(int(tri_counts[g])):
            gs.append(g); ps.append(p)
    for g in rng.choice(hall, 600):
        gs.append(g); ps.append(int(rng.integers(0, tri_counts[g])))
    bs = _bary_set(rng, 4)
    g = np.repeat(np.array(gs), len(bs)); p = np.repeat(np.array(ps), len(bs))
    uv = np.tile(bs, (len(gs), 1))
    return g, p, uv[:, 0], uv[:, 1]


def _gpu_hits(world):
    """Closest hits the GPU's own traversal finds: the primary rays of the frame (with their pixels) and random rays inside the hall."""
    ctx, pfd, rng = world["ctx"], world["pfds"][0], world["rng"]
    vi = pfd["camera_view_inverse"].reshape(4, 4).astype(np.float64)      # column-major: row 3 = translation
    vpi = pfd["camera_viewproj_inverse"].reshape(4, 4).astype(np.float64).T
    cam = vi[3, :3]
    ys, xs = np.mgrid[0:H:2, 0:W:2]
    xs, ys = xs.ravel(), ys.ravel()
    ndc = np.stack([(xs + 0.5) / W * 2 - 1, (ys + 0.5) / H * 2 - 1, np.ones_like(xs, np.float64), np.ones_like(xs, np.float64)], 1)
    pn = ndc @ vpi.T
    d = pn[:, :3] / pn[:, 3:4] - cam
    rays = np.zeros((len(xs), 8), f32)
    rays[:, :3], rays[:, 3], rays[:, 4:7], rays[:, 7] = cam, 1.0, d, 3.0e38
    st = ctx.bvh_stats()
    lo, hi = np.array(st.scene_min), np.array(st.scene_max)
    n = 20_000
    rr = np.zeros((n, 8), f32)
    rr[:, :3] = lo + (hi - lo) * rng.uniform(0.1, 0.9, (n, 3))
    rr[:, 3], rr[:, 4:7], rr[:, 7] = 0.01, rng.normal(size=(n, 3)), 1.0e4
    t, ids, uv = ctx.trace_explicit(np.concatenate([rays, rr]), any_hit=False)
    hit = t >= 0
    px = np.concatenate([xs, rng.integers(0, W, n)]); py = np.concatenate([ys, rng.integers(0, H, n)])
    return ids[hit, 0], ids[hit, 1], uv[hit, 0], uv[hit, 1], px[hit], py[hit], int(hit[:len(xs)].sum()), int(hit[len(xs):].sum())


@pytest.fixture(scope="module")
def hits(world):
    rng = world["rng"]
    g1, p1, u1, v1 = _synthetic_hits(world)
    x1, y1 = rng.integers(0, W, len(g1)), rng.integers(0, H, len(g1))
    at_corner = rng.choice(len(g1), len(g1) // 8, replace=False)               # the display corners
    x1[at_corner] = np.where(at_corner % 2 == 0, 0, W - 1)
    y1[at_corner] = np.where(at_corner % 4 < 2, 0, H - 1)
    g2, p2, u2, v2, x2, y2, n_primary, n_random = _gpu_hits(world)
    assert n_primary >= 5_000 and n_random >= 12_000
    rec = _records(np.concatenate([g1, g2]), np.concatenate([p1, p2]), np.concatenate([u1, u2]), np.concatenate([v1, v2]),
                   np.concatenate([x1, x2]), np.concatenate([y1, y2]))
    print(f"\n[hits] synthetic {len(g1)}, GPU-traced {len(g2)} ({n_primary} primary, {n_random} random in the hall)")
    return rec


def _coverage(sc, groups, rec):
    mat = sc.primitives["material"][rec["g"]]
    cnt = dict(records=len(rec),
               textured=int((mat["base_color_texture"] >= 0).sum()),
               normal_mapped=int((mat["normal_map"] >= 0).sum()),
               mr_textured=int((mat["metallic_roughness_texture"] >= 0).sum()),
               alpha_masked=int((mat["alpha_mask"] == 1).sum()),
               g_above_2048=int((rec["g"] > 2048).sum()),
               g_above_4096=int((rec["g"] > 4096).sum()),
               metallic_or_roughness_out_of_range=int(((mat["metallic_factor"] < 0) | (mat["metallic_factor"] > 1) |
                                                       (mat["roughness_factor"] < 0) | (mat["roughness_factor"] > 1)).sum()))
    for name, gs in groups.items():
        cnt["group_" + name] = int(np.isin(rec["g"], gs).sum())
    return cnt


KINDS = {"reflection": T.SHADE_REFLECTION, "gbuffer": T.SHADE_GBUFFER, "gbuffer_alpha": T.SHADE_GBUFFER_ALPHA,
         "raytraced": T.SHADE_RAYTRACED, "raytraced_alpha": T.SHADE_RAYTRACED_ALPHA, "anyhit_alpha": T.SHADE_ANYHIT_ALPHA}


@pytest.mark.parametrize("frame", [0, 1])
def test_hit_shading_bit_exact_on_identical_hits(world, hits, frame):
    sc, groups, ctx, osc = world["sc"], world["groups"], world["ctx"], world["osc"]
    pfd = world["pfds"][frame]
    ctx.update_per_frame_ubo(pfd)
    cov = _coverage(sc, groups, hits)
    out = {}
    for name, kind in KINDS.items():
        got, want = ctx.shade_hits(kind, hits), osc.shade_hits(pfd, kind, hits)
        if name == "gbuffer":
            # the documented NaN case: a normal-mapped hit whose tangent, made orthogonal to the normal, is exactly zero (the degenerate
            # frame) stores a NaN normal; its fp16 halves are compared as a class
            halves = [got[:, 1:3].copy().view(np.uint16), want[:, 1:3].copy().view(np.uint16)]      # [n, 4]: normal xyz, object id
            nan_g, nan_w = _is_nan16(halves[0]), _is_nan16(halves[1])
            assert (nan_g == nan_w).all() and not nan_w[:, 3].any(), f"frame {frame}: the two sides disagree on which normals are NaN"
            nan_rows = nan_w.any(axis=1)
            assert (sc.primitives["material"]["normal_map"][hits["g"][nan_rows]] >= 0).all(), "a NaN normal without a normal map"
            cov["gbuffer_nan_normal"] = int(nan_rows.sum())
            got, want = got.copy(), want.copy()
            halves[0][nan_g], halves[1][nan_w] = 0, 0
            got[:, 1:3], want[:, 1:3] = halves[0].view(np.uint32), halves[1].view(np.uint32)
        _same_bits(got, want, f"frame {frame} {name}")
        out[name] = got
    # branch coverage, shown rather than assumed
    gb_acc, rh_acc = out["gbuffer_alpha"][:, 0], out["anyhit_alpha"][:, 0]
    masked = sc.primitives["material"]["alpha_mask"][hits["g"]] == 1
    tie = np.isin(hits["g"], groups["alpha_cutoff_tie"])
    first_vertex = sc.primitives["vertex_offset"][hits["g"][tie]] + sc.indices[sc.primitives["index_offset"][hits["g"][tie]] + 3 * hits["pid"][tie]]
    tie[tie] = np.floor(sc.vertices["uv0"][first_vertex, 0] * 5).astype(int) == 1          # the texel whose alpha is the cutoff
    tie_texel = tie
    cov.update(alpha_rejected=int((gb_acc == 0).sum()), alpha_rejected_masked=int(((gb_acc == 0) & masked).sum()),
               alpha_rejected_zero=int(((gb_acc == 0) & ~masked).sum()), anyhit_rejected=int((rh_acc == 0).sum()),
               alpha_accepted_at_equality=int((tie & tie_texel & (gb_acc == 1)).sum()),
               anyhit_accepted_at_equality=int((tie & tie_texel & (rh_acc == 1)).sum()),
               no_direct_light=int((out["raytraced"][:, 0] == out["raytraced"][:, 1]).sum()))
    print(f"\n[hit shading, frame {frame}]", cov)
    need = dict(textured=20_000, normal_mapped=8_000, mr_textured=8_000, alpha_masked=2_000, g_above_2048=4_000, g_above_4096=1_000,
                metallic_or_roughness_out_of_range=1_000, alpha_rejected_masked=500, alpha_rejected_zero=300, anyhit_rejected=500,
                alpha_accepted_at_equality=50, anyhit_accepted_at_equality=50, no_direct_light=2_000, group_mirrored=400,
                group_rot_scale_tangent_w_neg=400, group_degenerate_frame=400)
    short = {k: (cov[k], v) for k, v in need.items() if cov[k] < v}
    assert not short, f"branches taken too rarely (count, needed): {short}"


def test_shade_hits_rejects_invalid_records(world):
    ctx, sc = world["ctx"], world["sc"]
    ctx.update_per_frame_ubo(world["pfds"][0])
    n_prims = len(sc.primitives)
    last = int(sc.primitives["index_count"][n_prims - 1] // 3)
    ok = _records([0, n_prims - 1], [0, last - 1], [0.2, 0.2], [0.3, 0.3])
    ctx.shade_hits(T.SHADE_GBUFFER, ok)
    for bad in (_records([n_prims], [0], [0.2], [0.3]), _records([n_prims - 1], [last], [0.2], [0.3]), _records([0xffffffff], [0], [0.0], [0.0])):
        for kind in (T.SHADE_REFLECTION, T.SHADE_GBUFFER, T.SHADE_ANYHIT_ALPHA):
            with pytest.raises(capi.VhrError, match="status -1"):
                ctx.shade_hits(kind, np.concatenate([ok, bad]))
    for slot in (len(sc.textures), 2047, 2048, 0xffffffff):
        with pytest.raises(capi.VhrError, match="status -1"):
            ctx.shade_hits(T.SHADE_TEXTURE, _records([0, slot], 0, [0.5, 0.5], [0.5, 0.5]))
    with pytest.raises(capi.VhrError, match="status -1"):
        ctx.shade_hits(7, ok)
    with capi.Context(16, 16) as c2:
        with pytest.raises(capi.VhrError, match="status -4"):                   # no per-frame constants
            c2.shade_hits(T.SHADE_TEXTURE, _records([0], 0, [0.5], [0.5]))
        c2.update_per_frame_ubo(world["pfds"][0])
        with pytest.raises(capi.VhrError, match="status -4"):                   # no geometry
            c2.shade_hits(T.SHADE_GBUFFER, ok)
