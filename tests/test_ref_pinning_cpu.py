"""CPU: pins the hand-written oracle (oracle/*.cpp) to oracle/_ref — the reference's OWN shader files compiled for the CPU
(oracle/make_ref.py reads the reference's data/shaders/*.{comp,rgen,rchit,rmiss,frag} + common.glsl + glsl_common.h at build time;
types and built-ins are the reference's vendored glm). Every comparison here is BIT FOR BIT: fp16 images as uint16, 8-bit images as
bytes, helper results as fp32 bit patterns.

Where the implementation is free (GLSL leaves normalize()/mat*vec evaluation order and NaN handling of max()/pow() open) both sides
follow one documented choice: glm's formulas for the former, the behaviour of the RT-capable GPUs the reference needs for the
latter (oracle/ref_shim.h).

oracle/_ref can only be built where the reference's sources are. Where the library is absent, every comparison is made against
tests/golden/ref_pinning_digests.json instead: the SHA-256 of each compared output on the same seeded inputs, so the check stays bit
exact. The digests were recorded from the oracle; its sources (oracle/*.cpp, oracle_common.h) are those of the last version that
passed all of these comparisons live against oracle/_ref. With the library present,
`VHR_RECORD_REF_DIGESTS=1 python -m pytest tests/test_ref_pinning_cpu.py` runs the live comparisons and rewrites the file.
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import helpers as Hh
import oracle_lib as O
import ref_lib as R
from vulkanhybridrenderer_b200 import camera, scenes
from vulkanhybridrenderer_b200 import types as T

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIGESTS = os.path.join(GOLDEN, "ref_pinning_digests.json")
LIVE = R.available()
RECORD = os.environ.get("VHR_RECORD_REF_DIGESTS") == "1"
_recorded = {}


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view({2: np.uint16, 4: np.uint32, 1: np.uint8}[a.dtype.itemsize])


def assert_same(a, b, what):
    a, b = bits(a), bits(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    bad = int(np.count_nonzero(a != b))
    assert bad == 0, f"{what}: {bad} of {a.size} values differ between oracle/ and oracle/_ref"


def digest(a):
    a = bits(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def _stored():
    with open(DIGESTS) as f:
        return json.load(f)["digests"]


def pinned(key, ours, theirs=None):
    """The oracle's output `ours` against oracle/_ref's for the same inputs: `theirs()` when the library is present (None: no live
    comparison, the stored digest is a drift guard only), else the stored digest of that output."""
    if LIVE and theirs is not None:
        assert_same(ours, theirs(), key)
    if RECORD:
        _recorded[key] = digest(ours)
    elif not LIVE:
        want = _stored().get(key)
        assert want is not None, f"{key}: no stored digest in {DIGESTS}"
        assert digest(ours) == want, f"{key}: the oracle's output differs from oracle/_ref's (stored digest)"


@pytest.fixture(scope="module", autouse=True)
def _record_digests():
    yield
    if RECORD:
        digests = {**(_stored() if os.path.exists(DIGESTS) else {}), **_recorded}
        with open(DIGESTS, "w") as f:
            json.dump({"what": "SHA-256 (dtype, shape, raw bytes) of each output tests/test_ref_pinning_cpu.py compares bit for bit between the oracle "
                               "and oracle/_ref, on that file's seeded inputs",
                       "digests": dict(sorted(digests.items()))}, f, indent=0)
            f.write("\n")


# ---- common.glsl + glsl_common.h ------------------------------------------------------------------------------------------------
def test_struct_sizes_from_the_reference_header():
    ours = np.array([T.PerFrameData.itemsize, T.Vertex.itemsize, 44, T.Primitive.itemsize, T.SVGFPushConstants.itemsize, 16, 4, 112], np.int32)
    pinned("struct sizes", ours, lambda: np.array([R.lib().vr_sizeof(which) for which in range(8)], np.int32))
    assert list(ours[:4]) == [584, 56, 44, 120]


def _rng_streams(seed_thread, random01, seeds, n):
    """Per seed: the state after seed_thread and after each of n random01 draws, and the n draws."""
    states, draws = np.zeros((len(seeds), n + 1), np.uint32), np.zeros((len(seeds), n), np.float32)
    for i, seed in enumerate(seeds):
        st = C.c_uint32(seed_thread(int(seed)))
        states[i, 0] = st.value
        for j in range(n):
            draws[i, j] = random01(C.byref(st))
            states[i, j + 1] = st.value
    return states, draws


def test_rng_known_answers_come_from_the_reference_text():
    """The KATs of SURVEY Appendix A.3 / tests/golden/rng_kat.npz were derived by hand in round 1; here common.glsl:47-76 itself runs."""
    OL = O.lib()
    kat = np.load(os.path.join(GOLDEN, "rng_kat.npz"))
    seeded = np.array([OL.vo_seed_thread(int(seed)) for seed in kat["seeds"]], np.uint32)
    assert np.array_equal(seeded, kat["states"])
    pinned("rng kat seed_thread", seeded, lambda: np.array([R.lib().vr_seed_thread(int(seed)) for seed in kat["seeds"]], np.uint32))
    _, draws = _rng_streams(int, OL.vo_random01, kat["states"], 8)
    assert_same(draws, kat["random01"], "random01 streams of the KAT states")
    pinned("rng kat random01", draws, lambda: _rng_streams(int, R.lib().vr_random01, kat["states"], 8)[1])
    seeds = np.random.default_rng(11).integers(0, 2**32, 2000, dtype=np.uint64)
    states, draws = _rng_streams(OL.vo_seed_thread, OL.vo_random01, seeds, 4)
    ref = _rng_streams(R.lib().vr_seed_thread, R.lib().vr_random01, seeds, 4) if LIVE else (None, None)
    pinned("rng random seeds states", states, lambda: ref[0])
    pinned("rng random seeds random01", draws, lambda: ref[1])
    assert np.all((draws >= 0.0) & (draws < 1.0))


def _sampling_helpers(L, p, us, dirs):
    cone, hemi, onb = np.zeros((len(us), 3), np.float32), np.zeros((len(us), 3), np.float32), np.zeros((len(dirs), 9), np.float32)
    for i, (u0, u1) in enumerate(us):
        getattr(L, p + "_uniform_sample_cone")(float(u0), float(u1), 0.999995, O._p(cone[i]))
        getattr(L, p + "_cosine_hemisphere")(float(u0), float(u1), O._p(hemi[i]))
    for i, d in enumerate(dirs):
        getattr(L, p + "_onb")(O._p(np.ascontiguousarray(d, np.float32)), O._p(onb[i]))
    return cone, hemi, onb


def test_sampling_helpers_bit_exact():
    rng = np.random.default_rng(5)
    us = rng.uniform(0, 1, (3000, 2)).astype(np.float32)
    dirs = rng.standard_normal((3000, 3)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    dirs = np.concatenate([dirs, np.array([[0, 0, -1], [0, 0, 1], [1e-4, 0, -0.99999994]], np.float32)])
    ours = _sampling_helpers(O.lib(), "vo", us, dirs)
    ref = _sampling_helpers(R.lib(), "vr", us, dirs) if LIVE else (None,) * 3
    for k, what in enumerate(("uniform_sample_cone", "uniform_sample_cosine_weighted_hemisphere", "onb_from_unit_vector")):
        pinned(what, ours[k], lambda: ref[k])


def _fp16_tables(L, p, xs):
    h2f = np.array([getattr(L, p + "_h2f")(h) for h in range(65536)], np.float32)
    h2f[np.isnan(h2f)] = np.nan            # any NaN is a match: one bit pattern for all of them
    return h2f, np.array([getattr(L, p + "_f2h")(float(x)) for x in xs], np.uint16)


def test_fp16_conversion_tables_agree():
    rng = np.random.default_rng(2)
    xs = np.concatenate([rng.standard_normal(20000).astype(np.float32) * np.float32(10.0) ** rng.integers(-9, 6, 20000).astype(np.float32),
                         np.array([0.0, -0.0, 65504.0, 65519.9, 65520.0, 1e-8, 5.96e-8, 2.98e-8, 2.9802322e-8, np.inf, -np.inf], np.float32)])
    h2f, f2h = _fp16_tables(O.lib(), "vo", xs)
    ref = _fp16_tables(R.lib(), "vr", xs) if LIVE else (None, None)
    pinned("fp16 h2f table", h2f, lambda: ref[0])
    pinned("fp16 f2h", f2h, lambda: ref[1])
    # numpy's float16 conversion is a third, independent implementation of round-to-nearest-even
    assert np.array_equal(f2h, xs.astype(np.float16).view(np.uint16))


def test_texture_unit_bit_exact_all_modes():
    """texture(textures[i], uv) of the shim (Vulkan LOD-0 formulas) vs the oracle's sampler: filters x address modes x UNORM / sRGB."""
    rng = np.random.default_rng(3)
    rgba = rng.integers(0, 256, (7, 5, 4), dtype=np.uint8)
    sc = scenes.sponza_like(500, seed=1, width=32, height=32, n_clutter=2)
    osc = O.OracleScene(sc)
    uvs = np.concatenate([rng.uniform(-2.5, 3.5, (400, 2)), np.array([[0, 0], [1, 1], [0.5, 0.5], [0.1, 0.9999999], [-1e-7, 1.0]])]).astype(np.float32)

    def ref_samples(fmt, mag, wu, wv):
        out = np.zeros((len(uvs), 4), np.float32)
        for i, (u, v) in enumerate(uvs):
            R.lib().vr_sample_rgba8(O._p(rgba), 5, 7, int(fmt), mag, mag, wu, wv, float(u), float(v), O._p(out[i]))
        return out
    for fmt in (T.VK_FORMAT_R8G8B8A8_UNORM, 43):
        for mag in (0, 1):
            for wu in range(4):
                for wv in range(4):
                    idx = osc.add_texture(rgba, fmt, (mag, mag, wu, wv))
                    ours = np.stack([osc.sample_texture(idx, u, v) for u, v in uvs])
                    pinned(f"texture fmt {fmt} filter {mag} wrap ({wu},{wv})", ours, lambda: ref_samples(fmt, mag, wu, wv))


# ---- shader passes ----------------------------------------------------------------------------------------------------------------
def _frames(W, H, tris, seed, n_frames, textured=False):
    sc = scenes.sponza_like(tris, seed=seed, width=W, height=H, n_clutter=12)
    if textured:
        sc = scenes.add_procedural_textures(sc, size=32)
    osc = O.OracleScene(sc)
    seq = camera.FrameSequencer(W, H, sc.light)
    cam = sc.camera
    for f in range(n_frames):
        if f:
            cam.set_pose(cam.position + np.array([0.06, 0.0, 0.02]), cam.yaw + 0.004, cam.pitch)
        pfd = seq.next(cam)
        yield sc, osc, pfd, osc.gbuffer(pfd, W, H)


@pytest.mark.parametrize("textured", [False, True])
@pytest.mark.parametrize("size", [(96, 64), (101, 59)])
def test_every_pass_of_the_hybrid_path_bit_exact_over_three_frames(size, textured):
    W, H = size
    so, sr = O.SvgfState(W, H), (R.SvgfState(W, H) if LIVE else None)
    sm = np.random.default_rng(1).uniform(0, 1, (32, 32)).astype(np.float32)
    for f, (sc, osc, pfd, g) in enumerate(_frames(W, H, 6000, 21, 3, textured)):
        tag = f"hybrid {W}x{H}{' textured' if textured else ''} frame {f}"
        a = osc.raygen(pfd, g["depth"], g["normals"])                                     # oracle: raygen.rgen restated
        b = R.raygen(sc, osc, pfd, g["depth"], g["normals"]) if LIVE else None            # the reference's raygen.rgen + miss + reflection_hit.rchit
        pinned(f"{tag} Raytraced Shadows and Ambient Occlusion", a["shadow_ao"], lambda: b["shadow_ao"])
        pinned(f"{tag} Raytraced Reflections", a["reflections"], lambda: b["reflections"])
        do, io, to = so.run(pfd, g["normals"], g["motion"], a["shadow_ao"])
        dr, ir, tr = sr.run(pfd, g["normals"], g["motion"], a["shadow_ao"]) if LIVE else (None,) * 3
        pinned(f"{tag} svgf.comp integrated", to, lambda: tr)
        pinned(f"{tag} five a-trous iterations", io, lambda: ir)
        pinned(f"{tag} Denoised (= iteration 3, SURVEY Q1)", do, lambda: dr)
        for k in range(5):
            pinned(f"{tag} persistent SVGF image {k}", so.image(k), lambda: sr.image(k))
        ra = O.ssao(pfd, g["depth"], g["normals"])
        pinned(f"{tag} ssao.comp", ra, lambda: R.ssao(pfd, g["depth"], g["normals"]))
        pinned(f"{tag} ssao_blur.comp", O.ssao_blur(pfd, ra), lambda: R.ssao_blur(pfd, ra))
        sa = O.ssr(pfd, g["albedo"], g["normals"], g["motion"], g["depth"])
        pinned(f"{tag} ssr.comp", sa, lambda: R.ssr(pfd, g["albedo"], g["normals"], g["motion"], g["depth"]))
        for modes in ((0, 0, 0), (1, 1, 1), (2, 2, 2), (0, 1, 2), (1, 0, 1)):
            for fmt in (T.VK_FORMAT_R16G16B16A16_SFLOAT, T.VK_FORMAT_B8G8R8A8_SRGB, T.VK_FORMAT_B8G8R8A8_UNORM):
                kw = dict(ssao_img=ra, ssr_img=sa, refl=a["reflections"], shadow_map=sm, out_format=fmt)
                x = O.composition(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], do, *modes, **kw)
                pinned(f"{tag} composition.frag modes {modes} format {fmt}", x,
                       lambda: R.composition(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], do, *modes, **kw))
            x = O.composition(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], a["shadow_ao"], *modes, refl=a["reflections"])
            pinned(f"{tag} composition.frag on the raw RG16F image, modes {modes}", x,
                   lambda: R.composition(pfd, g["albedo"], g["normals"], g["motion"], g["depth"], a["shadow_ao"], *modes, refl=a["reflections"]))


@pytest.mark.parametrize("step", [1, 2, 3, 4, 8, 16])
def test_atrous_on_worst_case_noise(step):
    W, H = 96, 64
    sc, osc, pfd, g = next(_frames(W, H, 6000, 21, 1))
    integ = Hh.noise_integrated(H, W, seed=2)
    pinned(f"a-trous step {step} on noise", O.svgf_atrous(pfd, g["normals"], integ, step), lambda: R.svgf_atrous(pfd, g["normals"], integ, step))
    # opposing normals: pow(negative, 128) must give weight 0 (SURVEY Q10), not C's (+1)
    flipped = g["normals"].copy()
    flipped[::2, :, :3] *= np.float16(-1.0)
    pinned(f"a-trous step {step}, opposing normals", O.svgf_atrous(pfd, flipped, integ, step), lambda: R.svgf_atrous(pfd, flipped, integ, step))


def test_temporal_with_random_history_and_large_motion():
    W, H = 120, 72
    it = _frames(W, H, 6000, 4, 2)
    sc, osc, pfd0, g0 = next(it)
    _, _, pfd1, g1 = next(it)
    rng = np.random.default_rng(7)
    rt = np.stack([rng.integers(0, 2, (H, W)), rng.integers(0, 3, (H, W)) * 0.5], -1).astype(np.float16)
    history = rng.uniform(0, 1, (H, W, 4)).astype(np.float16)
    moments = rng.uniform(0, 1, (H, W, 2)).astype(np.float16)
    for scale in (1.0, 8.0, -300.0):        # the last one throws most reprojections off screen
        motion = g1["motion"].copy()
        motion[..., :2] = (motion[..., :2].astype(np.float32) * scale).astype(np.float16)
        ai, am = O.svgf_temporal(pfd1, g1["normals"], motion, rt, g0["normals"], history, moments)
        bi, bm = R.svgf_temporal(pfd1, g1["normals"], motion, rt, g0["normals"], history, moments) if LIVE else (None, None)
        pinned(f"svgf.comp integrated, motion x{scale}", ai, lambda: bi)
        pinned(f"svgf.comp moments, motion x{scale}", am, lambda: bm)


def test_ssao_radius_and_sky_samples():
    W, H = 96, 64
    sc, osc, pfd, g = next(_frames(W, H, 6000, 21, 1))
    assert np.count_nonzero(g["depth"] == 0) > 0, "the frame should contain sky (samples that unproject to infinity / NaN)"
    for radius in (0.75, 0.2, 3.0):
        pinned(f"ssao.comp radius {radius}", O.ssao(pfd, g["depth"], g["normals"], radius), lambda: R.ssao(pfd, g["depth"], g["normals"], radius))


def test_golden_fixtures_are_outputs_of_the_reference_shaders():
    """tests/golden/hybrid_frames_96x64.npz and atrous_noise_96x64.npz: every shader-pass output stored there is reproduced by oracle/_ref
    from the stored inputs (tools/make_golden.py generates them from oracle/_ref). Without the library the oracle, which the tests above
    hold bit-identical to it, reproduces them instead."""
    z = np.load(os.path.join(GOLDEN, "hybrid_frames_96x64.npz"))
    W, H = 96, 64
    impl = R if LIVE else O

    class _Sc:
        vertices, indices, primitives, textures = z["vertices"], z["indices"], z["primitives"], []
    osc = O.OracleScene(_Sc)
    st = impl.SvgfState(W, H)
    for f in range(3):
        pfd = z[f"f{f}_pfd"]
        b = R.raygen(_Sc, osc, pfd, z[f"f{f}_depth"], z[f"f{f}_normals"]) if LIVE else osc.raygen(pfd, z[f"f{f}_depth"], z[f"f{f}_normals"])
        assert_same(b["shadow_ao"], z[f"f{f}_shadow_ao"], f"golden frame {f} shadow/AO")
        assert_same(b["reflections"], z[f"f{f}_reflections"], f"golden frame {f} reflections")
        den, iters, temporal = st.run(pfd, z[f"f{f}_normals"], z[f"f{f}_motion"], z[f"f{f}_shadow_ao"])
        assert_same(temporal, z[f"f{f}_temporal"], f"golden frame {f} temporal")
        assert_same(iters, z[f"f{f}_atrous"], f"golden frame {f} a-trous")
        assert_same(den, z[f"f{f}_denoised"], f"golden frame {f} denoised")
        raw = impl.ssao(pfd, z[f"f{f}_depth"], z[f"f{f}_normals"], 0.75)
        assert_same(raw, z[f"f{f}_ssao_raw"], f"golden frame {f} ssao raw")
        assert_same(impl.ssao_blur(pfd, raw), z[f"f{f}_ssao"], f"golden frame {f} ssao")
    n = np.load(os.path.join(GOLDEN, "atrous_noise_96x64.npz"))
    for s in (1, 2, 3, 4, 8, 16):
        assert_same(impl.svgf_atrous(n["pfd"], n["normals"], n["integ"], s), n[f"step{s}"], f"golden a-trous noise step {s}")
    t = np.load(os.path.join(GOLDEN, "textured_frame_96x64.npz"))
    assert_same(impl.ssr(t["pfd"], t["albedo"], t["normals"], t["motion"], t["depth"]), t["ssr"], "golden textured frame ssr")


@pytest.mark.parametrize("textured", [False, True])
def test_fully_raytraced_path_bit_exact(textured):
    """raytraced_render_path/{raygen.rgen, closesthit.rchit, miss.rmiss, shadow_miss.rmiss} (and the alpha-tested pipeline: raygen_test_alpha.rgen,
    closesthit_test_alpha.rchit, shadow_anyhit.rahit run as the any-hit stage of the oracle's traversal) compiled from the reference: the
    8-bit "RaytracedOutput" of the port is identical. The alpha-tested shaders index textures[base_color_texture] unconditionally, which is undefined
    for a material without a texture (index -1): there the port falls back to the base colour, so the comparison is on the textured primitives
    (without the library: the port's whole image against the digest recorded while it met that comparison)."""
    W, H = 96, 64
    for f, (sc, osc, pfd, g) in enumerate(_frames(W, H, 6000, 21, 2, textured)):
        tag = f"raytraced{' textured' if textured else ''} frame {f}"
        pinned(f"{tag} Raytracing Pipeline (opaque)", osc.raytraced(pfd, W, H, False), lambda: R.raytraced(sc, osc, pfd, W, H, False))
        a = osc.raytraced(pfd, W, H, True)
        ids = osc.gbuffer(pfd, W, H, want_ids=True)["ids"][..., 0]
        tex = sc.primitives["material"]["base_color_texture"]
        on_textured = np.where(ids >= 0, tex[np.clip(ids, 0, len(tex) - 1)] >= 0, True)      # sky pixels (miss.rmiss) count too
        if LIVE:
            b = R.raytraced(sc, osc, pfd, W, H, True)
            # `ids` comes from the G-buffer producer's primary ray, which is generated differently from this path's: on a silhouette pixel the two
            # may see different primitives, one of them untextured
            bad = np.any(a[on_textured] != b[on_textured], axis=-1)
            assert bad.sum() <= 3, f"frame {f} Raytracing Pipeline (alpha-tested): {int(bad.sum())} of {int(on_textured.sum())} pixels on textured primitives / sky differ"
        pinned(f"{tag} Raytracing Pipeline (alpha-tested)", a)
        if textured:
            assert on_textured.sum() > 0.4 * W * H
