"""GPU: the gathered output of a partitioned frame (VHR_OPT_OUTPUT_RANK). With the option set to p under a partition, every other
rank's composition draw stores its band a second time into rank p's RENDER_OUTPUT, so rank p ends with the whole frame of the
single-GPU draw, byte for byte, while every other rank keeps its band as before.

The ranks are contexts of ONE process on ONE GPU (peers attached by device pointer), as in tests/test_partition_gpu.py. Every rank
issues its passes before anything is downloaded: a download on a rank whose stream waits for a peer that has not issued yet would
block. In-process ranks stop at 3 (tests/test_partition_shadow_map_gpu.py says why); the two-process variant at the end runs
tools/time_partition_gather.py's parity check over real ranks."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import helpers as Hh
from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import multi_gpu as MG
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRGB, UNORM, HDR = T.VK_FORMAT_B8G8R8A8_SRGB, T.VK_FORMAT_B8G8R8A8_UNORM, T.VK_FORMAT_R16G16B16A16_SFLOAT
SHADER_PRESENT = "raytraced_render_path/composition.frag"
RT_OUT = "RaytracedOutput"
ERR_INVALID, ERR_STATE = -1, -4


def _scene(W, H):
    return scenes.sponza_like(20_000, seed=3, width=W, height=H, n_clutter=30)


def _poses(sc, W, H, n_frames):
    seq, cam, out = camera.FrameSequencer(W, H, sc.light), sc.camera, []
    for f in range(n_frames):
        if f:
            cam.set_pose(cam.position + np.array([0.05, 0.0, 0.01]), cam.yaw + 0.002, cam.pitch)
        out.append(seq.next(cam))
    return out


def _context(sc, W, H, **path_kw):
    ctx = capi.Context(W, H)
    ctx.load_scene(sc)
    ctx.set_option(capi.OPT_AO_SPP, 2)
    ctx.set_option(capi.OPT_TRACE_REFLECTIONS, 1)
    return ctx, HP.HybridRenderPath(ctx, W, H, **path_kw)


def _bytes(a):
    return a.view(np.uint8).reshape(a.shape[0], -1)


def _assert_rows(got, want, y0, y1, what):
    bad = _bytes(got)[y0:y1] != _bytes(want)[y0:y1]
    rows = np.nonzero(bad.any(axis=1))[0] + y0
    assert not bad.any(), f"{what}: {int(bad.sum())} mismatching bytes in rows [{y0},{y1}), rows {rows[:16].tolist()}"


def _outside(a, y0, y1):
    return np.concatenate([_bytes(a)[:y0], _bytes(a)[y1:]])


def _draw_hybrid(ctx, path, rtset, modes):
    g = path.gsets[0]
    ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH], HP.N_SHADOW_MAP, HP.N_SSAO, HP.N_SSR,
                          HP.N_DENOISED, path.rt_sets[rtset][1], HP.N_RENDER_OUTPUT])
    ctx.draw(HP.SHADER_COMPOSITION, modes)


class _Hybrid:
    """A single context and `world` partitioned ones rendering the camera-in hybrid frame: partitioned G-Buffer Pass, Raytrace + SVGF,
    SSAO, SSR, then composition (ray-traced shadows, SSAO, ray-traced reflections)."""
    MODES = (HP.SHADOW_MODE_RAYTRACED, HP.AO_MODE_SSAO, HP.REFLECTION_MODE_RAYTRACED)

    def __init__(self, world, fmt, output_rank, W=320):
        self.world, self.W, self.H = world, W, 64 * world + 17          # ragged last 8-row block and band
        self.sc = _scene(self.W, self.H)
        comp = dict(ssao=True, composition=fmt, shadow_map_size=(8, 8))
        self.ref_ctx, self.ref_path = _context(self.sc, self.W, self.H, **comp)
        self.ranks = [_context(self.sc, self.W, self.H, rt_sets=2, **comp) for _ in range(world)]
        self.ctxs, self.paths = [c for c, _ in self.ranks], [p for _, p in self.ranks]
        MG.setup_fused_partition_inprocess(self.ctxs, self.paths, motion_halo=24, exchange_gbuffer=True, output_rank=output_rank)
        self.bands = [MG.band_rows(self.H, world, r) for r in range(world)]

    def passes(self, pfd, rtset):
        """everything before the composition draw, on the single context and on every rank; returns the single context's output"""
        self.ref_ctx.update_per_frame_ubo(pfd)
        self.ref_path.gbuffer_pass()
        self.ref_path.frame(pfd)
        self.ref_path.ssao_passes()
        self.ref_path.ssr_pass()
        self.ref_path.composition_pass(*self.MODES, denoised=True)
        for ctx, path in self.ranks:
            ctx.update_per_frame_ubo(pfd)
            path.gbuffer_pass()
        for path in self.paths:
            path.frame(pfd, rtset=rtset)
        for path in self.paths:
            path.ssao_passes()
            path.ssr_pass()
        return self.ref_ctx.image_download(HP.N_RENDER_OUTPUT)

    def draw(self, rtset):
        """the composition draw on every rank; returns the kernels each one enqueued"""
        n0 = [c.kernel_launches for c in self.ctxs]
        for ctx, path in self.ranks:
            _draw_hybrid(ctx, path, rtset, self.MODES)
        return [c.kernel_launches - n for c, n in zip(self.ctxs, n0)]

    def close(self):
        for c in self.ctxs + [self.ref_ctx]:
            c.close()


def _gathered_frames(world, p, fmt, n_frames):
    fx = _Hybrid(world, fmt, p)
    try:
        assert [c.get_option(capi.OPT_OUTPUT_RANK) for c in fx.ctxs] == [p] * world
        pending = None           # (ticket, pinned host buffer, expected bytes) of the previous frame's read-back of rank p's output
        for f, pfd in enumerate(_poses(fx.sc, fx.W, fx.H, n_frames)):
            rtset = f & 1
            want = fx.passes(pfd, rtset)
            before = [None if r == p else ctx.image_download(HP.N_RENDER_OUTPUT) for r, ctx in enumerate(fx.ctxs)]
            # rank p's read-back of the previous frame may still be in flight: the draws must not overwrite its output before it ends
            assert fx.draw(rtset) == [1] * world, "the draw enqueues one kernel on every rank"
            if pending is not None:
                ticket, host, prev = pending
                fx.ctxs[p].wait_download(ticket)
                assert np.array_equal(host.numpy(), _bytes(prev).reshape(-1)), f"frame {f - 1}: rank {p}'s asynchronous read-back"
            for r, ctx in enumerate(fx.ctxs):
                got = ctx.image_download(HP.N_RENDER_OUTPUT)
                y0, y1 = fx.bands[r]
                if r == p:
                    _assert_rows(got, want, 0, fx.H, f"frame {f} output rank {p}/{world} fmt {fmt}: the whole frame")
                else:
                    _assert_rows(got, want, y0, y1, f"frame {f} rank {r}/{world} fmt {fmt}: its band")
                    assert np.array_equal(_outside(got, y0, y1), _outside(before[r], y0, y1)), f"frame {f} rank {r}: rows outside its band changed"
            host = torch.empty(want.nbytes, dtype=torch.uint8, pin_memory=True)
            pending = (fx.ctxs[p].image_download_rows_async(HP.N_RENDER_OUTPUT, host, 0, fx.H), host, want)
        fx.ctxs[p].wait_download(pending[0])
        assert np.array_equal(pending[1].numpy(), _bytes(pending[2]).reshape(-1))
    finally:
        fx.close()


@pytest.mark.parametrize("last", [False, True], ids=["rank0", "last_rank"])
@pytest.mark.parametrize("world", [2, 3])
def test_camera_in_frame_gathered_on_the_output_rank(world, last):
    _gathered_frames(world, world - 1 if last else 0, SRGB, 4)


@pytest.mark.parametrize("fmt", [SRGB, UNORM, HDR], ids=["B8G8R8A8_SRGB", "B8G8R8A8_UNORM", "R16G16B16A16_SFLOAT"])
def test_every_render_output_format(fmt):
    _gathered_frames(2, 1, fmt, 2)


def test_rasterised_shadow_frame_gathered():
    """partitioned G-Buffer Pass -> partitioned Shadow Map Pass -> SSAO -> composition (rasterised shadows, SSAO, no reflections)"""
    world, p, W, S = 2, 1, 320, (1000, 1000)
    H = 64 * world + 17
    sc = _scene(W, H)
    pts = Hh.world_triangles(sc).reshape(-1, 3)
    sc.light["projview"] = camera.fit_light_projview(sc.light["direction"][:3], pts.min(0), pts.max(0))
    comp = dict(ssao=True, composition=SRGB, shadow_map_size=S)
    modes = (HP.SHADOW_MODE_RASTERIZED, HP.AO_MODE_SSAO, HP.REFLECTION_MODE_OFF)
    ref_ctx, ref_path = _context(sc, W, H, **comp)
    ranks = [_context(sc, W, H, **comp) for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [q for _, q in ranks]
    try:
        MG.setup_fused_partition_inprocess(ctxs, paths, motion_halo=24, exchange_gbuffer=True, exchange_shadow_map=True, output_rank=p)
        for f, pfd in enumerate(_poses(sc, W, H, 3)):
            ref_ctx.update_per_frame_ubo(pfd)
            ref_path.gbuffer_pass()
            ref_path.shadow_map_pass()
            ref_path.ssao_passes()
            ref_path.composition_pass(*modes)
            for ctx, path in ranks:
                ctx.update_per_frame_ubo(pfd)
                path.gbuffer_pass()
            for path in paths:
                path.shadow_map_pass()
            for path in paths:
                path.ssao_passes()
            for path in paths:
                path.composition_pass(*modes)
            want = ref_ctx.image_download(HP.N_RENDER_OUTPUT)
            assert (ref_ctx.image_download(HP.N_SHADOW_MAP) > 0).mean() > 0.1
            _assert_rows(ctxs[p].image_download(HP.N_RENDER_OUTPUT), want, 0, H, f"frame {f} output rank {p}")
            y0, y1 = MG.band_rows(H, world, 0)
            _assert_rows(ctxs[0].image_download(HP.N_RENDER_OUTPUT), want, y0, y1, f"frame {f} rank 0")
    finally:
        for c in ctxs + [ref_ctx]:
            c.close()


def test_raytraced_render_path_gathered():
    """"Raytracing Pipeline" on each rank's band, then raytraced_render_path/composition.frag, for both pipelines"""
    world, p, W = 2, 0, 320
    H = 64 * world + 17
    sc = scenes.add_procedural_textures(_scene(W, H), size=32)

    def make():
        ctx = capi.Context(W, H)
        ctx.load_scene(sc)
        path = HP.HybridRenderPath(ctx, W, H, composition=SRGB)
        ctx.actualize_image(RT_OUT, UNORM)
        ctx.bind_pass_images([RT_OUT, HP.N_RENDER_OUTPUT])
        return ctx, path

    ref_ctx, _ = make()
    ranks = [make() for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [q for _, q in ranks]
    try:
        MG.setup_fused_partition_inprocess(ctxs, paths, output_rank=p)
        for f, pfd in enumerate(_poses(sc, W, H, 2)):
            for alpha in (0, 1):
                wants = []
                for ctx in [ref_ctx] + ctxs:
                    ctx.set_option(capi.OPT_RAYTRACED_ALPHA_TEST, alpha)
                    ctx.update_per_frame_ubo(pfd)
                    ctx.bind_pass_images([RT_OUT])
                    ctx.trace_rays(W, H, pipeline="Raytracing Pipeline")
                    ctx.bind_pass_images([RT_OUT, HP.N_RENDER_OUTPUT])
                    n0 = ctx.kernel_launches
                    ctx.draw(SHADER_PRESENT, ())
                    wants.append(ctx.kernel_launches - n0)
                assert wants == [1] * (world + 1)
                want = ref_ctx.image_download(HP.N_RENDER_OUTPUT)
                assert (_bytes(want) != 0).mean() > 0.5
                _assert_rows(ctxs[p].image_download(HP.N_RENDER_OUTPUT), want, 0, H, f"frame {f} alpha {alpha} output rank {p}")
                y0, y1 = MG.band_rows(H, world, 1)
                _assert_rows(ctxs[1].image_download(HP.N_RENDER_OUTPUT), want, y0, y1, f"frame {f} alpha {alpha} rank 1")
    finally:
        for c in ctxs + [ref_ctx]:
            c.close()


def test_option_back_off_under_the_partition():
    """gathered frame 0, then the option back to -1: each rank's draw writes only its band; the output rank's rows outside its band keep
    frame 0's bytes"""
    world, p = 2, 1
    fx = _Hybrid(world, SRGB, p)
    try:
        pfds = _poses(fx.sc, fx.W, fx.H, 2)
        want0 = fx.passes(pfds[0], 0)
        assert fx.draw(0) == [1] * world
        _assert_rows(fx.ctxs[p].image_download(HP.N_RENDER_OUTPUT), want0, 0, fx.H, "frame 0 gathered")
        for ctx in fx.ctxs:
            ctx.set_option(capi.OPT_OUTPUT_RANK, -1)
        want1 = fx.passes(pfds[1], 1)
        before = [ctx.image_download(HP.N_RENDER_OUTPUT) for ctx in fx.ctxs]
        assert fx.draw(1) == [1] * world
        assert not np.array_equal(_bytes(want0), _bytes(want1)), "the two frames must differ"
        for r, ctx in enumerate(fx.ctxs):
            got = ctx.image_download(HP.N_RENDER_OUTPUT)
            y0, y1 = fx.bands[r]
            _assert_rows(got, want1, y0, y1, f"frame 1 rank {r}: its band")
            assert np.array_equal(_outside(got, y0, y1), _outside(before[r], y0, y1)), f"rank {r}: rows outside its band changed"
        y0, y1 = fx.bands[p]
        assert np.array_equal(_outside(fx.ctxs[p].image_download(HP.N_RENDER_OUTPUT), y0, y1), _outside(want0, y0, y1))
    finally:
        fx.close()


@pytest.mark.parametrize("shader", ["hybrid", "raytraced"])
def test_single_context_ignores_the_option(shader):
    """without a partition the option changes no byte and no launch count"""
    W, H = 320, 145
    sc = _scene(W, H)
    pfd = _poses(sc, W, H, 1)[0]
    outs = []
    for value in (-1, 0, 3):
        ctx, path = _context(sc, W, H, ssao=True, composition=SRGB, shadow_map_size=(8, 8))
        try:
            ctx.set_option(capi.OPT_OUTPUT_RANK, value)
            assert ctx.get_option(capi.OPT_OUTPUT_RANK) == value
            ctx.update_per_frame_ubo(pfd)
            path.gbuffer_pass()
            if shader == "hybrid":
                path.frame(pfd)
                path.ssao_passes()
                path.ssr_pass()
                n0 = ctx.kernel_launches
                path.composition_pass(*_Hybrid.MODES, denoised=True)
            else:
                ctx.actualize_image(RT_OUT, UNORM)
                ctx.bind_pass_images([RT_OUT])
                ctx.trace_rays(W, H, pipeline="Raytracing Pipeline")
                ctx.bind_pass_images([RT_OUT, HP.N_RENDER_OUTPUT])
                n0 = ctx.kernel_launches
                ctx.draw(SHADER_PRESENT, ())
            assert ctx.kernel_launches - n0 == 1
            outs.append(ctx.image_download(HP.N_RENDER_OUTPUT))
        finally:
            ctx.close()
    assert (_bytes(outs[0]) != 0).any()
    for o in outs[1:]:
        assert np.array_equal(_bytes(o), _bytes(outs[0]))


def test_errors():
    """Out-of-range values; an output rank outside the partition (every rank fails); a missing attachment (the draw is issued on the
    misconfigured rank only: the output rank would pass its checks and wait for a signal nobody writes). Every error comes before
    anything is enqueued: afterwards every context synchronises, clears the partition and renders."""
    world, W = 2, 320
    H = 64 * world + 17
    sc = _scene(W, H)
    ranks = [_context(sc, W, H, ssao=True, composition=SRGB, shadow_map_size=(8, 8)) for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [q for _, q in ranks]
    try:
        for bad in (-2, capi.MAX_RANKS, 1 << 40):
            with pytest.raises(capi.VhrError, match=rf"vhr status {ERR_INVALID}: output rank"):
                ctxs[0].set_option(capi.OPT_OUTPUT_RANK, bad)
        assert ctxs[0].get_option(capi.OPT_OUTPUT_RANK) == -1
        with pytest.raises(ValueError, match="not a rank"):
            MG.setup_fused_partition_inprocess(ctxs, paths, output_rank=world)
        MG.setup_fused_partition_inprocess(ctxs, paths)                  # RENDER_OUTPUT of rank 0 attached nowhere
        pfd = _poses(sc, W, H, 1)[0]
        for ctx in ctxs:
            ctx.update_per_frame_ubo(pfd)
        # the output rank is not a rank of the partition: every rank fails, nothing is enqueued
        for ctx, path in ranks:
            ctx.set_option(capi.OPT_OUTPUT_RANK, world)
            with pytest.raises(capi.VhrError, match=rf"vhr status {ERR_INVALID}: composition: VHR_OPT_OUTPUT_RANK {world} is not a rank"):
                _draw_hybrid(ctx, path, 0, _Hybrid.MODES)
        # rank 1 without rank 0's render output attached: the draw on rank 1 only
        for ctx in ctxs:
            ctx.set_option(capi.OPT_OUTPUT_RANK, 0)
        with pytest.raises(capi.VhrError, match=rf"vhr status {ERR_STATE}: composition: the render output \('{HP.N_RENDER_OUTPUT}'\) has no image of rank 0"):
            _draw_hybrid(ctxs[1], paths[1], 0, _Hybrid.MODES)
        ctxs[1].actualize_image(RT_OUT, UNORM)
        ctxs[1].bind_pass_images([RT_OUT, HP.N_RENDER_OUTPUT])
        with pytest.raises(capi.VhrError, match=rf"vhr status {ERR_STATE}: raytraced composition: the render output \('{HP.N_RENDER_OUTPUT}'\) has no image of rank 0"):
            ctxs[1].draw(SHADER_PRESENT, ())
        for ctx in ctxs:
            ctx.synchronize()
        for ctx, path in ranks:
            ctx.clear_partition()
            path.gbuffer_pass()
            n0 = ctx.kernel_launches
            _draw_hybrid(ctx, path, 0, _Hybrid.MODES)
            assert ctx.kernel_launches - n0 == 1
            ctx.synchronize()
            assert (_bytes(ctx.image_download(HP.N_RENDER_OUTPUT)) != 0).any()
    finally:
        for c in ctxs:
            c.close()


def test_setup_needs_the_render_output():
    world, W = 2, 320
    H = 64 * world + 17
    sc = _scene(W, H)
    ranks = [_context(sc, W, H) for _ in range(world)]          # no composition: RENDER_OUTPUT does not exist
    try:
        with pytest.raises(ValueError, match="RENDER_OUTPUT"):
            MG.setup_fused_partition_inprocess([c for c, _ in ranks], [q for _, q in ranks], output_rank=0)
    finally:
        for c, _ in ranks:
            c.close()


def _gpu_count():
    try:
        import ctypes
        cuda = ctypes.CDLL("libcuda.so.1")
        n = ctypes.c_int(0)
        return n.value if cuda.cuInit(0) == 0 and cuda.cuDeviceGetCount(ctypes.byref(n)) == 0 else 0
    except OSError:
        return 0


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs (cuDeviceGetCount < 2)")
def test_gathered_frame_over_two_processes_is_bit_exact(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tools", "time_partition_gather.py"), "--parity-only", "--width", "960", "--height", "544", "--tris", "60000",
           "--frames", "4", "--output-rank", "1", "--out", str(tmp_path / "t.json")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "PARITY OK (bit-exact)" in r.stdout
