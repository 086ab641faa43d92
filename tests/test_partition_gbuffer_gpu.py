"""GPU: the G-Buffer Pass under the fused partition. Every rank traces its own rows and stores them into every rank's G-buffer, so
each rank holds the whole G-buffer of the single-GPU pass, byte for byte, and the partitioned frame can be driven from a camera
with nothing uploaded.

The ranks are contexts of ONE process on ONE GPU (peers attached by device pointer), as in tests/test_partition_gpu.py; the
two-process variant at the end runs tools/time_partition_camera_in.py's parity check over real ranks."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import multi_gpu as MG

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GBUFFER = (HP.N_ALBEDO, HP.N_NORMALS, HP.N_MOTION, HP.N_DEPTH)


def _scene(kind, W, H):
    sc = scenes.sponza_like(20_000, seed=3, width=W, height=H, n_clutter=30)
    return scenes.add_procedural_textures(sc, size=32) if kind == "textured" else sc


def _context(sc, W, H, **path_kw):
    ctx = capi.Context(W, H)
    ctx.load_scene(sc)
    ctx.set_option(capi.OPT_AO_SPP, 2)
    ctx.set_option(capi.OPT_TRACE_REFLECTIONS, 1)
    return ctx, HP.HybridRenderPath(ctx, W, H, **path_kw)


def _poses(sc, W, H, n_frames):
    """pfd of each frame of a moving camera"""
    seq, cam, out = camera.FrameSequencer(W, H, sc.light), sc.camera, []
    for f in range(n_frames):
        if f:
            cam.set_pose(cam.position + np.array([0.05, 0.0, 0.01]), cam.yaw + 0.002, cam.pitch)
        out.append(seq.next(cam))
    return out


@pytest.mark.parametrize("scene", ["plain", "textured"])
@pytest.mark.parametrize("world,ray_block_rows", [(2, 8), (3, 8), (2, 0)])
def test_partitioned_gbuffer_is_the_whole_single_gpu_gbuffer_on_every_rank(world, ray_block_rows, scene):
    W, H, n_frames = 320, 64 * world + 17, 4            # ragged last 8-row block and band
    sc = _scene(scene, W, H)
    ref_ctx, ref_path = _context(sc, W, H)
    ranks = [_context(sc, W, H) for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [p for _, p in ranks]
    try:
        MG.setup_fused_partition_inprocess(ctxs, paths, ray_block_rows=ray_block_rows, exchange_gbuffer=True)
        for f, pfd in enumerate(_poses(sc, W, H, n_frames)):
            for ctx, path in [(ref_ctx, ref_path)] + ranks:
                ctx.update_per_frame_ubo(pfd)
                path.gbuffer_pass()
            want = {k: ref_ctx.image_download(k) for k in GBUFFER}
            assert (want[HP.N_DEPTH] > 0).mean() > 0.3 and (want[HP.N_DEPTH] == 0).any(), "the frame must show geometry and sky"
            for r, ctx in enumerate(ctxs):
                for k in GBUFFER:
                    got = ctx.image_download(k)
                    bad = got.view(np.uint8) != want[k].view(np.uint8)
                    assert not bad.any(), (f"frame {f} rank {r}/{world} {k}: {int(bad.sum())} mismatching bytes, rows "
                                           f"{np.nonzero(bad.reshape(H, -1).any(axis=1))[0][:16].tolist()}")
    finally:
        for c in ctxs + [ref_ctx]:
            c.close()


@pytest.mark.parametrize("gbuffer_sets", [1, 2])
@pytest.mark.parametrize("world", [2, 3])
def test_camera_in_partitioned_frame_matches_single_context(world, gbuffer_sets):
    """partitioned G-Buffer Pass -> Raytrace + SVGF -> SSAO -> SSR -> composition (ray-traced shadows, SSAO, ray-traced reflections), with
    nothing uploaded. SSR reads G-buffer rows far outside the band. One G-buffer set (every pass first waits for all ranks) and two
    alternating sets (no leading wait) give the reference's bytes."""
    W, H, n_frames = 320, 64 * world + 17, 4
    sc = _scene("plain", W, H)
    comp = dict(ssao=True, composition=HP.T.VK_FORMAT_B8G8R8A8_SRGB, shadow_map_size=(8, 8))
    ref_ctx, ref_path = _context(sc, W, H, **comp)
    ranks = [_context(sc, W, H, gbuffer_sets=gbuffer_sets, rt_sets=2, **comp) for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [p for _, p in ranks]
    try:
        halo = 24
        MG.setup_fused_partition_inprocess(ctxs, paths, motion_halo=halo, exchange_gbuffer=True)
        bands = [MG.band_rows(H, world, r) for r in range(world)]
        for f, pfd in enumerate(_poses(sc, W, H, n_frames)):
            gset, rtset = f % gbuffer_sets, f & 1
            ref_ctx.update_per_frame_ubo(pfd)
            ref_path.gbuffer_pass()
            motion = ref_ctx.image_download(HP.N_MOTION)
            assert MG.required_motion_halo(float(np.abs(motion[..., 1].astype(np.float32)).max()), H) <= halo
            ref_path.frame(pfd)
            ref_path.ssao_passes()
            ref_path.ssr_pass()
            ref_path.composition_pass(0, 1, 0, denoised=True)
            # every rank issues the same calls; nothing blocks on the host, the streams order themselves through the flag words
            for ctx, path in ranks:
                ctx.update_per_frame_ubo(pfd)
                path.gbuffer_pass(gset)
            for path in paths:
                path.frame(pfd, gset=gset, rtset=rtset)
            for path in paths:
                path.ssao_passes(gset)
                path.ssr_pass(gset)
            for ctx, path in ranks:
                g = path.gsets[gset]
                ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH], HP.N_SHADOW_MAP, HP.N_SSAO, HP.N_SSR,
                                      HP.N_DENOISED, path.rt_sets[rtset][1], HP.N_RENDER_OUTPUT])
                ctx.draw(HP.SHADER_COMPOSITION, (0, 1, 0))
            want = {k: ref_ctx.image_download(n) for k, n in (("rt", HP.N_RT), ("refl", HP.N_REFL), ("den", HP.N_DENOISED), ("ssao", HP.N_SSAO),
                                                              ("ssr", HP.N_SSR), ("out", HP.N_RENDER_OUTPUT))}
            for r, (ctx, path) in enumerate(ranks):
                y0, y1 = bands[r]
                got = {"rt": ctx.image_download(path.rt_sets[rtset][0]), "refl": ctx.image_download(path.rt_sets[rtset][1]),
                       "den": ctx.image_download(HP.N_DENOISED), "ssao": ctx.image_download(HP.N_SSAO), "ssr": ctx.image_download(HP.N_SSR),
                       "out": ctx.image_download(HP.N_RENDER_OUTPUT)}
                for k in want:
                    bad = int((got[k][y0:y1].view(np.uint8) != want[k][y0:y1].view(np.uint8)).sum())
                    assert bad == 0, f"frame {f} rank {r}/{world} sets {gbuffer_sets} image {k}: {bad} mismatching bytes in rows [{y0},{y1})"
    finally:
        for c in ctxs + [ref_ctx]:
            c.close()


def test_partitioned_gbuffer_without_exchanged_images_fails_on_every_rank():
    """Without the G-buffer images of the other ranks attached the pass is refused before anything is enqueued: every rank fails the
    same way and no stream is left waiting for a peer (the contexts still synchronise and render afterwards)."""
    world, W = 2, 320
    H = 64 * world + 17
    sc = _scene("plain", W, H)
    ranks = [_context(sc, W, H) for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [p for _, p in ranks]
    try:
        MG.setup_fused_partition_inprocess(ctxs, paths, exchange_gbuffer=False)
        pfd = _poses(sc, W, H, 1)[0]
        for ctx, path in ranks:
            ctx.update_per_frame_ubo(pfd)
            with pytest.raises(capi.VhrError, match=rf"vhr status {-4}: G-buffer pass: binding 0 \('{HP.N_ALBEDO}'\) has no image of rank \d"):
                path.gbuffer_pass()
        for ctx in ctxs:
            ctx.synchronize()
        for ctx, path in ranks:   # the unpartitioned pass still runs on each context
            ctx.clear_partition()
            path.gbuffer_pass()
            ctx.synchronize()
            assert (ctx.image_download(HP.N_DEPTH) > 0).any()
    finally:
        for c in ctxs:
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
def test_camera_in_partition_over_two_processes_is_bit_exact(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tools", "time_partition_camera_in.py"), "--parity-only", "--width", "960", "--height", "544", "--tris", "60000",
           "--frames", "4", "--out", str(tmp_path / "t.json")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "PARITY OK (bit-exact)" in r.stdout
