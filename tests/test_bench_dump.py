"""bench.py --dump-outputs: the images the last timed step computed, as float32 .npy files within a 64 MB budget, so that two builds can be
compared output for output on identical inputs."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

import bench
from vulkanhybridrenderer_b200 import hybrid_path as HP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _loop(W, H, refl, fif=1, frame_no=7):
    """The attributes of bench.GpuFrameLoop that dump_outputs reads; channel 0 of every image holds the pixel index."""
    rt_sets = [(HP.N_RT, HP.N_REFL), (HP.N_RT + " [1]", HP.N_REFL + " [1]")][:fif]
    images = {}
    for k, (rt, rf) in enumerate([(HP.N_DENOISED, None)] + rt_sets):
        for name, ch in ((rt, 4 if rt == HP.N_DENOISED else 2), (rf, 4)):
            if name is not None:
                a = np.full((H, W, ch), k + 0.5, np.float32)
                a[..., 0] = np.arange(W * H, dtype=np.float32).reshape(H, W)
                images[name] = a
    ctx = types.SimpleNamespace(image_download=lambda name: images[name].copy())
    return types.SimpleNamespace(HP=HP, W=W, H=H, refl=refl, fif=fif, frame_no=frame_no, ctx=ctx,
                                 path=types.SimpleNamespace(rt_sets=rt_sets)), images


def test_dump_of_a_1080p_frame_is_whole(tmp_path):
    loop, images = _loop(1920, 1080, refl=0)
    bench.dump_outputs(str(tmp_path), loop, 0, 1)
    assert sorted(os.listdir(tmp_path)) == ["denoised_shadow_ao.npy", "raytraced_shadow_ao.npy"]
    for name, img in (("denoised_shadow_ao", HP.N_DENOISED), ("raytraced_shadow_ao", HP.N_RT)):
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == np.float32
        np.testing.assert_array_equal(a, images[img])


def test_dump_over_the_budget_is_one_seeded_pixel_sample(tmp_path):
    # 4K with reflections (10 channels, 332 MB as float32); two frames in flight, last frame odd: the second ray-output set
    loop, images = _loop(3840, 2160, refl=1, fif=2, frame_no=8)
    bench.dump_outputs(str(tmp_path), loop, 1, 2)
    names = ["denoised_shadow_ao_rank1.npy", "raytraced_reflections_rank1.npy", "raytraced_shadow_ao_rank1.npy"]
    assert sorted(os.listdir(tmp_path)) == names
    got = [np.load(tmp_path / n) for n in names]
    assert sum(a.nbytes for a in got) * 2 <= bench.DUMP_BUDGET_BYTES
    idx = got[0][:, 0]
    assert np.all(np.diff(idx) > 0) and len(idx) > 100_000
    for a, img in zip(got, (HP.N_DENOISED, HP.N_REFL + " [1]", HP.N_RT + " [1]")):
        assert a.dtype == np.float32 and a.shape[1] == images[img].shape[2]
        np.testing.assert_array_equal(a, images[img].reshape(-1, a.shape[1])[idx.astype(np.int64)])
    again = tmp_path / "again"
    bench.dump_outputs(str(again), loop, 1, 2)
    np.testing.assert_array_equal(np.load(again / names[0]), got[0])


def test_views64_steps_must_be_whole_batches():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "views64_1080p_3Mtri", "--steps", "100"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "multiple of 64" in r.stderr


def _bench_dump(out, steps, warmup, fif):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", str(steps), "--warmup", str(warmup),
                        "--frames-in-flight", str(fif), "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["ms_per_step"] > 0
    assert sorted(os.listdir(out)) == ["denoised_shadow_ao.npy", "raytraced_shadow_ao.npy"]
    return np.load(out / "denoised_shadow_ao.npy"), np.load(out / "raytraced_shadow_ao.npy")


@pytest.mark.gpu
def test_bench_dumps_its_last_step(tmp_path):
    """Both runs end on the same frame (warm-up + timed steps = 8) on the same seeded inputs; the second has two frames in flight, so its
    last frame's ray output sits in the second image set. A dump of any other frame, or of the wrong set, would differ."""
    den, rt = _bench_dump(tmp_path / "a", 5, 3, 1)
    assert den.dtype == rt.dtype == np.float32 and den.shape == (184, 320, 4) and rt.shape == (184, 320, 2)
    assert np.isfinite(rt).all() and (rt[..., 0] > 0).any() and (rt[..., 0] == 0).any()      # lit and shadowed pixels both
    assert np.any(np.nan_to_num(den[..., :2]) != 0)
    den2, rt2 = _bench_dump(tmp_path / "b", 4, 4, 2)
    assert np.array_equal(rt, rt2)
    assert np.array_equal(den, den2, equal_nan=True)
