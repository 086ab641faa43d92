"""GPU parity: Alchemy SSAO + 13x13 blur (through the C-ABI) vs the CPU oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

import exact_helpers_lib as E
import helpers as Hh
import checker as O
from vulkanhybridrenderer_b200 import capi
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu
F4 = T.VK_FORMAT_R16G16B16A16_SFLOAT


def _groups(n):
    return n // 8 + (n % 8 != 0)


def _libm_sincos(x):
    """sinf / cosf of the C library: what the oracle's std::sin(float) / std::cos(float) call."""
    libm = C.CDLL("libm.so.6")
    for f in (libm.sinf, libm.cosf):
        f.restype, f.argtypes = C.c_float, [C.c_float]
    flat = x.reshape(-1)
    return (np.array([libm.sinf(float(v)) for v in flat], np.float32).reshape(x.shape),
            np.array([libm.cosf(float(v)) for v in flat], np.float32).reshape(x.shape))


def _cuda_sincos(x):
    flat = torch.from_numpy(np.ascontiguousarray(x.reshape(-1))).cuda()
    s, c = torch.empty_like(flat), torch.empty_like(flat)
    E.call("eh_sincos_eval", flat, flat.numel(), s, c)
    torch.cuda.synchronize()
    return s.cpu().numpy().reshape(x.shape), c.cpu().numpy().reshape(x.shape)


def _explain_mismatches(pfd, raw, ref, what):
    """Every SSAO pixel whose fp16 bits differ from the checker's must own a sample angle on which CUDA's sincosf and the C library's
    sinf / cosf disagree (the kernel is otherwise written in the oracle's operations and order); such pixels are at most 1e-3 of the
    image. Returns the number of explained pixels."""
    bad = np.argwhere(np.any(raw.view(np.uint16) != ref.view(np.uint16), axis=-1))
    H, W = raw.shape[:2]
    if len(bad):
        ang = Hh.ssao_sample_angles(pfd, bad[:, 1], bad[:, 0])
        (cs, cc), (ls, lc) = _cuda_sincos(ang), _libm_sincos(ang)
        differs = np.any((cs.view(np.uint32) != ls.view(np.uint32)) | (cc.view(np.uint32) != lc.view(np.uint32)), axis=-1)
        unexplained = bad[~differs]
    else:
        unexplained = bad
    print(f"[ssao] {what}: {len(bad)} of {H * W} pixels differ from the checker, {len(bad) - len(unexplained)} explained by sincosf")
    assert len(unexplained) == 0, f"{what}: pixels (y, x) that differ with no sincosf disagreement: {unexplained[:8].tolist()}"
    assert len(bad) <= 1e-3 * H * W, (what, len(bad))
    return len(bad)


SSAO_CASES = [
    pytest.param((320, 184), 0.75, "default", id="size0-0.75"),
    pytest.param((203, 117), 2.0, "default", id="size1-2.0"),
] + [pytest.param((203, 117), 2.0, cam, id=f"{cam}-203x117") for cam in Hh.CAMERA_CASES[1:]] + [
    pytest.param((203, 117), 2.0, "narrow_fov", id="narrow_fov-203x117"),
    pytest.param((203, 117), 2.0, "mirrored", id="mirrored-203x117"),
    pytest.param((203, 117), 1.0e4, "default", id="radius1e4-203x117"),
    pytest.param((1, 37), 2.0, "default", id="1x37"),
    pytest.param((2, 3), 2.0, "default", id="2x3"),
    pytest.param((7, 5), 2.0, "default", id="7x5"),
    pytest.param((9, 65), 2.0, "jitter", id="9x65-jitter"),
]


@pytest.mark.parametrize("size,radius,cam", SSAO_CASES)
def test_ssao_and_blur(size, radius, cam):
    W, H = size
    sc, osc, pfd, g = Hh.camera_case(cam, W, H)
    inv = pfd["camera_proj_inverse"].reshape(-1)
    # the host's range check must choose the general unprojection (ssao_kernel<false, ...>): coefficients out of range, or a negative
    # m00, whose sparse path would divide a -0 dividend (div_exact_flag_bounded takes +0 only)
    if cam == "narrow_fov":
        assert abs(inv[0]) < 2.0 ** -14 and abs(inv[5]) < 2.0 ** -14
    if cam == "mirrored":
        assert inv[0] < 0
    if radius > 1e3:                 # most samples land more than 2^14 texels away: the general tap path and several periods of REPEAT
        d = g["depth"].astype(np.float64)
        lit = d > 0
        reach = radius * d[lit] * abs(float(inv[11])) * W     # radius / |P.z| * W, P.z = -1 / (m23 depth) (column-major index 11)
        assert np.mean(reach > 2 ** 15) > 0.5
    ref_raw = O.ssao(pfd, g["depth"], g["normals"], radius)
    ref_blur = O.ssao_blur(pfd, ref_raw)
    r0, r1 = H // 4, H - H // 4
    with capi.Context(W, H) as ctx:
        ctx.update_per_frame_ubo(pfd)
        ctx.actualize_image(Hh.N_NORMALS, F4); ctx.actualize_image(Hh.N_DEPTH, T.VK_FORMAT_D32_SFLOAT)
        ctx.actualize_image(Hh.N_SSAO_RAW, F4); ctx.actualize_image(Hh.N_SSAO, F4)
        ctx.image_upload(Hh.N_NORMALS, g["normals"]); ctx.image_upload(Hh.N_DEPTH, g["depth"])
        ctx.bind_pass_images([Hh.N_NORMALS, Hh.N_DEPTH, Hh.N_SSAO_RAW])
        ctx.dispatch("hybrid_render_path/ssao.comp", _groups(W), _groups(H), 1, np.array([radius], np.float32))
        raw = ctx.image_download(Hh.N_SSAO_RAW)
        # blur the ORACLE's raw image so the blur kernel is judged on identical inputs
        ctx.image_upload(Hh.N_SSAO_RAW, ref_raw)
        ctx.bind_pass_images([Hh.N_SSAO_RAW, Hh.N_SSAO])
        ctx.dispatch("hybrid_render_path/ssao_blur.comp", _groups(W), _groups(H), 1, np.array([radius], np.float32))
        blur = ctx.image_download(Hh.N_SSAO)
        # a row band (multi-GPU split) computes the full frame's bits on its rows and writes nothing else
        ctx.image_upload(Hh.N_SSAO_RAW, np.full((H, W, 4), 7.0, np.float16))
        ctx.bind_pass_images([Hh.N_NORMALS, Hh.N_DEPTH, Hh.N_SSAO_RAW])
        ctx.set_option(capi.OPT_ROW_BEGIN, r0); ctx.set_option(capi.OPT_ROW_END, r1)
        ctx.dispatch("hybrid_render_path/ssao.comp", _groups(W), _groups(H), 1, np.array([radius], np.float32))
        band = ctx.image_download(Hh.N_SSAO_RAW)
    what = f"ssao raw {W}x{H} r={radius} camera {cam}"
    Hh.assert_parity(raw, ref_raw, what, max_abs=0.05)
    _explain_mismatches(pfd, raw, ref_raw, what)
    Hh.assert_parity(blur, ref_blur, f"ssao blur {W}x{H} camera {cam}")
    assert np.array_equal(band[r0:r1].view(np.uint16), raw[r0:r1].view(np.uint16))
    assert np.all(band[:r0].astype(np.float32) == 7.0) and np.all(band[r1:].astype(np.float32) == 7.0)
    ao = ref_raw[..., 0].astype(np.float32)
    assert np.any((ao > 0) & (ao < 0.99)), f"{what}: no occluded pixel in the reference (degenerate case)"
    if W * H > 1000:
        assert float(np.std(ao)) > 0.01, f"{what}: degenerate SSAO test image"
