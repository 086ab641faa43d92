"""GPU: the Shadow Map Pass under the fused partition. Every rank rasterises the 8-row blocks of the map dealt to it (block b to rank
b % world) and stores them into every rank's map, so each rank holds the whole map of the single-GPU pass, bit for bit.

The ranks are contexts of ONE process on ONE GPU (peers attached by device pointer), as in tests/test_partition_gpu.py. Every rank
issues its pass before anything is downloaded: a download on a rank whose stream waits for a peer that has not issued yet would
block. The two-process variant at the end runs tools/time_partition_shadow_map.py's parity check over real ranks."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import helpers as Hh
import shadow_map_lib as SM
from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import multi_gpu as MG
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D32 = T.VK_FORMAT_D32_SFLOAT
SIZES = [(512, 512), (1000, 1000), (517, 301)]


def _fitted(sc):
    p = Hh.world_triangles(sc).reshape(-1, 3)
    return camera.fit_light_projview(sc.light["direction"][:3], p.min(0), p.max(0))


def _window(sc, window):
    return camera.light_projview(sc.light["direction"][:3]) if window == "reference" else _fitted(sc)


def _pfd(sc, projview, W=64, H=48):
    light = sc.light.copy()
    light["projview"] = projview
    return camera.FrameSequencer(W, H, light).next(sc.camera)


def _map_name(size):
    return f"Map {size[0]}x{size[1]}"


class _Ranks:
    """`world` contexts with the same geometry and maps, partitioned in-process; `attach(r, q)` attaches rank q's maps to rank r.
    The display extent is 64 x 64 world, the least a partition's bands allow."""

    def __init__(self, sc, world, sizes):
        self.world, self.sizes = world, sizes
        self.W, self.H = 64, 64 * world
        self.ctxs = []
        for _ in range(world):
            ctx = capi.Context(self.W, self.H)
            ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
            for s in sizes:
                ctx.actualize_image(_map_name(s), D32, *s)
            self.ctxs.append(ctx)
        L = capi.lib()
        for r, ctx in enumerate(self.ctxs):
            for q, octx in enumerate(self.ctxs):
                if q != r:
                    capi._check(L.vhr_sync_attach_peer_pointer(ctx._h, q, L.vhr_sync_device_ptr(octx._h)))
        bands = [MG.band_rows(self.H, world, r)[0] for r in range(world)] + [self.H]
        for r, ctx in enumerate(self.ctxs):
            ctx.set_partition(world, r, bands)

    def attach(self, r, q):
        L = capi.lib()
        for s in self.sizes:
            n = _map_name(s)
            capi._check(L.vhr_image_attach_peer_pointer(self.ctxs[r]._h, n.encode(), q, self.ctxs[q].image_info(n)[0]))

    def attach_all(self):
        for r in range(self.world):
            for q in range(self.world):
                if q != r:
                    self.attach(r, q)

    def render(self, pfd, size):
        """every rank issues its pass, then every rank's map is downloaded"""
        for ctx in self.ctxs:
            ctx.update_per_frame_ubo(pfd)
            ctx.bind_pass_images([_map_name(size)])
            ctx.shadow_map_pass()
        return [ctx.image_download(_map_name(size)) for ctx in self.ctxs]

    def close(self):
        for c in self.ctxs:
            c.close()


def _single(sc, pfd, size):
    with capi.Context(64, 48) as ctx:
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.actualize_image("Shadow Map", D32, *size)
        ctx.update_per_frame_ubo(pfd)
        ctx.bind_pass_images(["Shadow Map"])
        ctx.shadow_map_pass()
        return ctx.image_download("Shadow Map")


def _assert_bits(got, want, what):
    bad = got.view(np.uint32) != want.view(np.uint32)
    rows = np.nonzero(bad.any(axis=1))[0]
    print(f"[partition shadow map] {what}: {int(bad.sum())} of {want.size} texels differ, {int(np.sum(want > 0))} covered")
    assert not bad.any(), f"{what}: {int(bad.sum())} texels differ, rows {rows[:16].tolist()}"


def _check_ranks(maps, want, what):
    for r, got in enumerate(maps):
        _assert_bits(got, want, f"{what}, rank {r} of {len(maps)}")


@pytest.mark.parametrize("world", [2, 3])
def test_every_rank_holds_the_single_gpu_map(world):
    """In-process ranks stop at 3, as in the other partition tests: eight contexts whose streams wait on each other's flag words
    share the device's hardware queues, and a wait queued ahead of the signal it needs can then stall them."""
    sc = scenes.sponza_like(20_000, seed=3, n_clutter=30)
    ranks = _Ranks(sc, world, SIZES)
    try:
        ranks.attach_all()
        for window in ("reference", "fitted"):
            pfd = _pfd(sc, _window(sc, window))
            for size in SIZES:
                want = _single(sc, pfd, size)
                assert (want > 0).any()
                _assert_bits(want, SM.shadow_map(sc, pfd, *size), f"single context {size} {window}")
                _check_ranks(ranks.render(pfd, size), want, f"{size} {window}")
    finally:
        ranks.close()


def test_tiny_map_with_ranks_that_own_no_rows():
    """8 x 8: one block of rows, dealt to rank 0; ranks 1 and 2 own nothing and still take part in both waits"""
    sc = scenes.tiny_scene()
    size = (8, 8)
    ranks = _Ranks(sc, 3, [size])
    try:
        ranks.attach_all()
        for window in ("reference", "fitted"):
            pfd = _pfd(sc, _window(sc, window))
            want = _single(sc, pfd, size)
            _assert_bits(want, SM.shadow_map(sc, pfd, *size), f"single context 8x8 {window}")
            assert (want > 0).any()
            for _ in range(2):
                _check_ranks(ranks.render(pfd, size), want, f"8x8 {window}")
    finally:
        ranks.close()


def test_sponza_4096_two_ranks():
    sc = scenes.sponza_like(260_000)
    size = (4096, 4096)
    ranks = _Ranks(sc, 2, [size])
    try:
        ranks.attach_all()
        for window in ("reference", "fitted"):
            pfd = _pfd(sc, _window(sc, window))
            want = SM.shadow_map(sc, pfd, *size)
            _check_ranks(ranks.render(pfd, size), want, f"sponza 260k 4096^2 {window}")
    finally:
        ranks.close()


class _Soup:
    """explicit world-space triangles: one primitive, identity transform (as tests/test_shadow_map_cpu.py)"""

    def __init__(self, tris):
        tris = np.asarray(tris, np.float32).reshape(-1, 3, 3)
        self.vertices = np.zeros(3 * len(tris), T.Vertex)
        self.vertices["pos"] = tris.reshape(-1, 3)
        self.indices = np.arange(3 * len(tris), dtype=np.uint32)
        self.primitives = np.zeros(1, T.Primitive)
        self.primitives["transform"] = np.eye(4, dtype=np.float32)
        self.primitives["index_count"] = 3 * len(tris)
        for k in ("base_color_texture", "metallic_roughness_texture", "normal_map"):
            self.primitives["material"][k] = -1          # untextured: the GPU context checks every named texture


def _texel_pfd(W, H):
    """world (x, y) -> map coordinates (x, y) exactly, z -> depth"""
    m = np.array([[2.0 / W, 0, 0, -1], [0, 2.0 / H, 0, -1], [0, 0, 1, 0], [0, 0, 0, 1]])
    pfd = np.zeros((), T.PerFrameData)
    pfd["directional_light"]["projview"] = np.asarray(camera.to_glm(m), np.float32).reshape(4, 4)
    return pfd


@pytest.mark.parametrize("world", [2, 3])
def test_guard_band_triangles(world):
    """Triangles reaching beyond the +-2^20-texel guard band go through the clip kernel; under the partition each rank clips them
    and shades only its own rows."""
    size = W, H = 61, 45
    big = 2.0 ** 22
    z = np.float32([0.25, 0.25 + big * 1e-7, 0.25 + big * 2e-7])
    tris = [
        [(8.0, 8.0, z[0]), (8.0 + big, 8.0, z[1]), (8.0, 8.0 + big, z[2])],              # beyond the band on both axes
        [(-big, 3.5, 0.5), (40.0, 3.5, 0.5), (40.0, 30.25, 0.75)],                         # beyond it on the left only
        [(20.0, -big, 0.9), (55.0, 40.0, 0.2), (2.0, 41.0, 0.6)],                          # above it only
        [(30.0, 20.0, 0.4), (34.0, 20.0, 0.4), (30.0, 24.0, 0.4)],                         # a small one inside the map
    ]
    sc = _Soup(tris)
    pfd = _texel_pfd(W, H)
    want = SM.shadow_map(sc, pfd, W, H)
    assert (want > 0).mean() > 0.5
    _assert_bits(_single(sc, pfd, size), want, "single context, guard band")
    ranks = _Ranks(sc, world, [size])
    try:
        ranks.attach_all()
        _check_ranks(ranks.render(pfd, size), want, "guard band")
    finally:
        ranks.close()


def test_consecutive_frames_leave_no_stale_rows():
    """fitted window, reference window, zero projview: after each frame every rank's map is the single-context map (after the third,
    all zero). A clear that wiped a peer's rows, or rows left from the previous frame, would show."""
    sc = scenes.sponza_like(20_000, seed=3, n_clutter=30)
    size = (517, 301)
    ranks = _Ranks(sc, 3, [size])
    try:
        ranks.attach_all()
        for f, pv in enumerate((_fitted(sc), camera.light_projview(sc.light["direction"][:3]), np.zeros((4, 4), np.float32))):
            pfd = _pfd(sc, pv)
            want = _single(sc, pfd, size)
            assert (want > 0).any() == (f < 2)
            _check_ranks(ranks.render(pfd, size), want, f"frame {f}")
    finally:
        ranks.close()


def test_geometry_that_grows_under_the_partition():
    """A larger scene between partitioned passes makes every rank's scratch grow inside the pass, after an earlier rank's stream already
    waits for this rank's signal: the outgrown buffers are retired, not freed (no device synchronisation), and the maps stay exact."""
    small, large = scenes.sponza_like(20_000, seed=3, n_clutter=30), scenes.sponza_like(260_000, seed=5)
    size = (1000, 1000)
    ranks = _Ranks(small, 3, [size])
    try:
        ranks.attach_all()
        for sc in (small, large, small):
            for ctx in ranks.ctxs:
                ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
            pfd = _pfd(sc, _fitted(sc))
            _check_ranks(ranks.render(pfd, size), _single(sc, pfd, size), f"{sc.num_triangles} triangles")
    finally:
        ranks.close()


def test_partitioned_pass_enqueues_one_launch_more():
    """the single-GPU pass: setup, the scan's two kernels, tile, clip (5); the partitioned pass adds the push (6)"""
    sc = scenes.sponza_like(20_000, seed=3, n_clutter=30)
    size = (1000, 1000)
    pfd = _pfd(sc, _fitted(sc))
    ranks = _Ranks(sc, 2, [size])
    try:
        ranks.attach_all()
        ranks.render(pfd, size)                      # the first partitioned call may also load the kernels
        n0 = [c.kernel_launches for c in ranks.ctxs]
        ranks.render(pfd, size)
        assert [c.kernel_launches - n for c, n in zip(ranks.ctxs, n0)] == [6, 6]
    finally:
        ranks.close()


def test_missing_attachments():
    """The map attached for some other ranks but not all: every rank fails with VHR_ERR_STATE naming the missing rank, before any
    flag word is written; the contexts still synchronise, and once the attachments are complete the pass runs partitioned. With
    nothing attached every rank renders the whole map (5 launches), the same bits."""
    sc = scenes.sponza_like(20_000, seed=3, n_clutter=30)
    size = (517, 301)
    pfd = _pfd(sc, _fitted(sc))
    want = _single(sc, pfd, size)
    world = 3
    ranks = _Ranks(sc, world, [size])
    try:
        n0 = [c.kernel_launches for c in ranks.ctxs]
        _check_ranks(ranks.render(pfd, size), want, "nothing attached (replicated)")
        assert [c.kernel_launches - n for c, n in zip(ranks.ctxs, n0)] == [5] * world
        for r in range(world):
            ranks.attach(r, (r + 1) % world)         # rank (r + 2) % world is missing
        for r, ctx in enumerate(ranks.ctxs):
            ctx.update_per_frame_ubo(pfd)
            ctx.bind_pass_images([_map_name(size)])
            missing = (r + 2) % world
            with pytest.raises(capi.VhrError, match=rf"vhr status {-4}: Shadow Map Pass: binding 0 \('{_map_name(size)}'\) has no image of rank {missing}"):
                ctx.shadow_map_pass()
        for ctx in ranks.ctxs:
            ctx.synchronize()
        for r in range(world):
            ranks.attach(r, (r + 2) % world)
        n0 = [c.kernel_launches for c in ranks.ctxs]
        _check_ranks(ranks.render(pfd, size), want, "attachments completed")
        assert all(c.kernel_launches - n >= 6 for c, n in zip(ranks.ctxs, n0))
    finally:
        ranks.close()


def _poses(sc, W, H, n_frames):
    seq, cam, out = camera.FrameSequencer(W, H, sc.light), sc.camera, []
    for f in range(n_frames):
        if f:
            cam.set_pose(cam.position + np.array([0.05, 0.0, 0.01]), cam.yaw + 0.002, cam.pitch)
        out.append(seq.next(cam))
    return out


@pytest.mark.parametrize("world", [2, 3])
def test_camera_in_rasterised_shadow_frame_matches_single_context(world):
    """partitioned G-Buffer Pass -> partitioned Shadow Map Pass -> SSAO -> composition (rasterised shadows, SSAO, no reflections) from a
    moving camera: every rank's band of RENDER_OUTPUT is the single context's, byte for byte."""
    W, H, n_frames, S = 320, 64 * world + 17, 3, (1000, 1000)
    sc = scenes.sponza_like(20_000, seed=3, width=W, height=H, n_clutter=30)
    sc.light["projview"] = _fitted(sc)                   # a window that holds the whole hall, so the frame shows shadows
    comp = dict(ssao=True, composition=T.VK_FORMAT_B8G8R8A8_SRGB, shadow_map_size=S)
    modes = (HP.SHADOW_MODE_RASTERIZED, HP.AO_MODE_SSAO, HP.REFLECTION_MODE_OFF)

    def make():
        ctx = capi.Context(W, H)
        ctx.load_scene(sc)
        return ctx, HP.HybridRenderPath(ctx, W, H, **comp)

    ref_ctx, ref_path = make()
    ranks = [make() for _ in range(world)]
    ctxs, paths = [c for c, _ in ranks], [p for _, p in ranks]
    try:
        MG.setup_fused_partition_inprocess(ctxs, paths, motion_halo=24, exchange_gbuffer=True, exchange_shadow_map=True)
        bands = [MG.band_rows(H, world, r) for r in range(world)]
        for f, pfd in enumerate(_poses(sc, W, H, n_frames)):
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
            want_map = ref_ctx.image_download(HP.N_SHADOW_MAP)
            assert (want_map > 0).mean() > 0.1
            for r, ctx in enumerate(ctxs):
                y0, y1 = bands[r]
                got = ctx.image_download(HP.N_RENDER_OUTPUT)
                bad = int((got[y0:y1].view(np.uint8) != want[y0:y1].view(np.uint8)).sum())
                assert bad == 0, f"frame {f} rank {r}/{world}: {bad} mismatching bytes of RENDER_OUTPUT in rows [{y0},{y1})"
                _assert_bits(ctx.image_download(HP.N_SHADOW_MAP), want_map, f"frame {f} rank {r} map")
    finally:
        for c in ctxs + [ref_ctx]:
            c.close()


def _gpu_count():
    try:
        import ctypes
        cuda = ctypes.CDLL("libcuda.so.1")
        n = ctypes.c_int(0)
        return n.value if cuda.cuInit(0) == 0 and cuda.cuDeviceGetCount(ctypes.byref(n)) == 0 else 0
    except OSError:
        return 0


@pytest.mark.parametrize("world", [2, 8])          # 8 = VHR_MAX_RANKS: the push kernel's whole peer table
def test_partitioned_shadow_map_over_processes_is_bit_exact(tmp_path, world):
    """one process per GPU over CUDA IPC: every rank's partitioned 4096^2 map against its replicated one (tools/time_partition_shadow_map.py)"""
    if _gpu_count() < world:
        pytest.skip(f"needs {world} GPUs (cuDeviceGetCount < {world})")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tools", "time_partition_shadow_map.py"), "--parity-only", "--tris", "60000", "--out", str(tmp_path / "t.json")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "PARITY OK (bit-exact)" in r.stdout
