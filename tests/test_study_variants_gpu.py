"""The study switches that DESIGN and the kernels describe as computing the default's bits do: VHR_SSAO_VARIANT 1, 2 and 16,
VHR_SSAO_BLUR_VARIANT=1, VHR_SSR_SKIP=1 and VHR_SSR_VARIANT=1 with each VHR_SSR_REGION.

The library reads each switch once per process, so every variant runs in a child python with the switch in its environment; the child
writes its images as .npy files and the names of the kernels that ran (torch.profiler), and the parent checks that the switch took
effect and compares the images with the default's bit for bit. Both the default camera (sparse inverse projection: ssao_kernel<true, V>,
SSR step skipping) and a jittered one (ssao_kernel<false, V>) are rendered. Run as a script, this file is the child."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

W, H = 61, 37                    # ragged: neither a multiple of 8 nor of the blur's 64 x 32 tile; above SSR's 16-pixel skipping limit
SSR_PARAMS = (8.0, 0.1, 0.5, 4)
VARIANTS = ([("VHR_SSAO_VARIANT", v) for v in ("1", "2", "16")] + [("VHR_SSAO_BLUR_VARIANT", "1"), ("VHR_SSR_SKIP", "1")] +
            [("VHR_SSR_VARIANT=1 VHR_SSR_REGION", r) for r in ("21", "22", "41", "42", "81", "82", "44")])


def _child(out_dir):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "tests"), os.path.join(root, "oracle")]
    import json
    import torch
    import helpers as Hh
    from vulkanhybridrenderer_b200 import capi
    from vulkanhybridrenderer_b200 import hybrid_path as HP
    from vulkanhybridrenderer_b200 import types as T
    F4 = T.VK_FORMAT_R16G16B16A16_SFLOAT
    noise = np.random.default_rng(3).uniform(0, 1, (H, W, 4)).astype(np.float16)
    out = {}
    torch.cuda.init()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        # the default camera (sparse inverse: ssao_kernel<true, V>, SSR step skipping applies) and a jittered one (ssao_kernel<false, V>)
        for cam in ("default", "jitter"):
            sc, osc, pfd, g = Hh.camera_case(cam, W, H)
            with capi.Context(W, H) as ctx:
                ctx.update_per_frame_ubo(pfd)
                for name, fmt in Hh.GBUF_IMAGES.items():
                    ctx.actualize_image(name, fmt)
                for name in (Hh.N_SSAO_RAW, Hh.N_SSAO, HP.N_SSR):
                    ctx.actualize_image(name, F4)
                ctx.image_upload(HP.N_ALBEDO, g["albedo"]); ctx.image_upload(HP.N_NORMALS, g["normals"])
                ctx.image_upload(HP.N_MOTION, g["motion"]); ctx.image_upload(HP.N_DEPTH, g["depth"])
                ctx.bind_pass_images([Hh.N_NORMALS, Hh.N_DEPTH, Hh.N_SSAO_RAW])
                ctx.dispatch("hybrid_render_path/ssao.comp", HP.groups(W), HP.groups(H), 1, np.array([2.0], np.float32))
                out[f"{cam}_ssao"] = ctx.image_download(Hh.N_SSAO_RAW)
                ctx.bind_pass_images([HP.N_ALBEDO, HP.N_NORMALS, HP.N_MOTION, HP.N_DEPTH, HP.N_SSR])
                n0 = ctx.kernel_launches
                ctx.dispatch(HP.SHADER_SSR, HP.groups(W), HP.groups(H), 1, np.array(SSR_PARAMS, T.SSRPushConstants))
                out[f"{cam}_ssr_launches"] = np.array(ctx.kernel_launches - n0)
                out[f"{cam}_ssr"] = ctx.image_download(HP.N_SSR)
                # the blur of a fixed noise image: whole image, a partial dispatch, a row band (each over a preset output)
                ctx.image_upload(Hh.N_SSAO_RAW, noise)
                ctx.bind_pass_images([Hh.N_SSAO_RAW, Hh.N_SSAO])
                for what, groups, rows in (("blur", (HP.groups(W), HP.groups(H)), None), ("blur_partial", (5, 3), None),
                                           ("blur_band", (HP.groups(W), HP.groups(H)), (9, 30))):
                    ctx.image_upload(Hh.N_SSAO, np.full((H, W, 4), 7.0, np.float16))
                    if rows:
                        ctx.set_option(capi.OPT_ROW_BEGIN, rows[0]); ctx.set_option(capi.OPT_ROW_END, rows[1])
                    ctx.dispatch("hybrid_render_path/ssao_blur.comp", *groups, 1, np.array([2.0], np.float32))
                    out[f"{cam}_{what}"] = ctx.image_download(Hh.N_SSAO)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    with open(os.path.join(out_dir, "kernels.json"), "w") as f:
        json.dump(sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}), f)


def _run(tmp, env_extra):
    d = tmp / ("_".join(f"{k}{v}" for k, v in env_extra.items()) or "default")
    d.mkdir()
    env = dict(os.environ)
    for k in [k for k in env if k.startswith("VHR_SSAO") or k.startswith("VHR_SSR")]:
        del env[k]
    env.update(env_extra)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(d)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    kernels = json.loads((d / "kernels.json").read_text())
    return {f[:-4]: np.load(d / f) for f in os.listdir(d) if f.endswith(".npy")}, kernels


def _tpl(name, *args):
    """Pattern of a demangled template kernel name: demanglers print an int / bool argument as 16 or (int)16, true or (bool)1."""
    def arg(a):
        if isinstance(a, bool):
            return rf"(\(bool\))?({'true|1' if a else 'false|0'})"
        return rf"(\(int\))?{a}"
    return name + "<" + r",\s*".join(arg(a) for a in args) + ">"


def _expected_kernels(switch, value):
    """Kernel-name patterns that show the switch took effect, and patterns of the default kernels it replaces."""
    if switch == "VHR_SSAO_VARIANT":
        v = int(value)
        return [_tpl("ssao_kernel", True, v), _tpl("ssao_kernel", False, v)], [_tpl("ssao_kernel", True, 0), _tpl("ssao_kernel", False, 0)]
    if switch == "VHR_SSAO_BLUR_VARIANT":
        return [r"ssao_blur_kernel\("], [r"ssao_blur_tile_kernel"]
    if switch == "VHR_SSR_SKIP":
        return [r"depth_tiles_kernel"], []
    tx, ty, g = {"21": (2, 1, 8), "22": (2, 1, 4), "41": (4, 1, 8), "42": (4, 1, 4), "81": (4, 2, 8), "82": (4, 2, 4), "44": (2, 2, 4)}[value]
    return [_tpl("ssr_refill_kernel", tx, ty, g)], [r"ssr_kernel\("]


@pytest.fixture(scope="module")
def default_run(tmp_path_factory):
    images, kernels = _run(tmp_path_factory.mktemp("variants"), {})
    names = "\n".join(kernels)
    for k in (_tpl("ssao_kernel", True, 0), _tpl("ssao_kernel", False, 0), r"ssao_blur_tile_kernel", r"ssr_kernel\("):
        assert re.search(k, names), (k, kernels)
    assert not re.search(r"depth_tiles_kernel|ssr_refill_kernel", names), kernels
    return images, kernels


@pytest.mark.gpu
@pytest.mark.parametrize("switch,value", VARIANTS, ids=[f"{k.replace(' ', '-')}={v}" for k, v in VARIANTS])
def test_study_switch_gives_the_default_bits(switch, value, default_run, tmp_path):
    default_images, _ = default_run
    env = dict(kv.split("=") for kv in switch.split()[:-1])
    env[switch.split()[-1]] = value
    got, kernels = _run(tmp_path, env)
    names = "\n".join(kernels)
    want, gone = _expected_kernels(switch.split()[-1], value)
    for k in want:
        assert re.search(k, names), f"{env}: the switch did not take effect ({k} never ran): {kernels}"
    for k in gone:
        assert not re.search(k, names), f"{env}: the default kernel {k} still ran: {kernels}"
    if switch == "VHR_SSR_SKIP":        # the tile pre-pass runs for the default camera only (the bound needs a sparse inverse)
        assert int(got["default_ssr_launches"]) == int(default_images["default_ssr_launches"]) + 1
    assert sorted(got) == sorted(default_images)
    for k, ref in default_images.items():
        if k.endswith("_launches"):
            continue
        assert np.array_equal(got[k].view(np.uint16), ref.view(np.uint16)), f"{env}: {k} differs on {int(np.sum(np.any(got[k].view(np.uint16) != ref.view(np.uint16), axis=-1)))} pixels"
    for cam in ("default", "jitter"):
        blur_partial = default_images[f"{cam}_blur_partial"].astype(np.float32)
        assert np.all(blur_partial[24:] == 7.0) and np.all(blur_partial[:, 40:] == 7.0) and not np.any(blur_partial[:24, :40] == 7.0)
        blur_band = default_images[f"{cam}_blur_band"].astype(np.float32)
        assert np.all(blur_band[:9] == 7.0) and np.all(blur_band[30:] == 7.0)
        assert np.array_equal(default_images[f"{cam}_blur_band"][9:30].view(np.uint16), default_images[f"{cam}_blur"][9:30].view(np.uint16))


if __name__ == "__main__":
    _child(sys.argv[1])
