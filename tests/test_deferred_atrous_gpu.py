"""Deferred a-trous dispatch (vhr_dispatch of svgf_atrous_filter.comp): the kernel runs when something can observe its output and not at
all when its output is overwritten unread. Every image a caller can read holds what the immediate launch leaves; the reference's last
iteration (step 16, overwritten by the next frame's iteration 0) costs no launch."""
import ctypes as C

import numpy as np
import pytest

import checker as O
import helpers as Hh
from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import types as T

pytestmark = pytest.mark.gpu

F4 = T.VK_FORMAT_R16G16B16A16_SFLOAT
W, H = 256, 144
ATROUS = "hybrid_render_path/svgf_atrous_filter.comp"


def _groups(n):
    return n // 8 + (n % 8 != 0)


def _eager(ctx):
    """A context whose a-trous dispatches launch at once: a second queue exists."""
    ctx.select_queue(1)
    ctx.select_queue(0)
    return ctx


class BenchFrames:
    """bench.py's frame loop at a small size: two G-buffer sets of two camera poses rendered up front, then frames alternating between
    them with the frame index advancing (HybridRenderPath.frame, copy-free blits on)."""

    def __init__(self, eager=False):
        self.sc = scenes.sponza_like(20000, seed=3, width=W, height=H, n_clutter=40)
        cam = self.sc.camera
        poses = [(cam.position, cam.yaw, cam.pitch), (cam.position + np.array([0.05, 0.0, 0.01]), cam.yaw + 0.002, cam.pitch)]
        self.ctx = capi.Context(W, H)
        if eager:
            _eager(self.ctx)
        self.ctx.update_geometry(self.sc.vertices, self.sc.indices, self.sc.primitives)
        self.path = HP.HybridRenderPath(self.ctx, W, H, gbuffer_sets=2, blit_alias=True)
        seq = camera.FrameSequencer(W, H, self.sc.light)
        self.pfds = [None, None]
        for s in (1, 0, 1):
            cam.set_pose(*poses[s])
            pfd = seq.next(cam)
            g = self.path.gsets[s]
            self.ctx.update_per_frame_ubo(pfd)
            self.ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
            self.ctx.gbuffer_pass(W, H)
            self.pfds[s] = pfd
        self.k = 0

    def frame(self):
        s = self.k & 1
        pfd = self.pfds[s]
        pfd["frame_index"] = 3 + self.k
        self.k += 1
        self.path.frame(pfd, gset=s)
        return s, pfd

    def svgf_images(self):
        """Every image the SVGF pass keeps: both integrated slots, previous normals, history, moments, Denoised."""
        pc = self.path.pc
        slots = {"integrated0": pc["integrated_shadow_and_ao"][0], "integrated1": pc["integrated_shadow_and_ao"][1],
                 "prev_normals": pc["prev_frame_normals_and_object_ids"], "history": pc["shadow_and_ao_history"],
                 "moments": pc["shadow_and_ao_moments_history"]}
        out = {k: self.ctx.storage_image_download(int(v)) for k, v in slots.items()}
        out["denoised"] = self.ctx.image_download(HP.N_DENOISED)
        return out

    def denoised_async(self):
        """Denoised through the download queue: no device pointer, no context synchronise."""
        host = np.empty((H, W, 4), np.float16)
        self.ctx.wait_download(self.ctx.image_download_async(HP.N_DENOISED, host))
        return host

    def close(self):
        self.ctx.close()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint16)


def test_bit_identity_with_and_without_read_backs():
    """Eight bench-style frames three ways: reading every SVGF image after every frame (each deferred dispatch is launched by the read),
    reading only Denoised (the last iteration is never launched), and with immediate launches. Denoised agrees bit for bit across all
    three, every image of the first agrees bit for bit with the immediate run, and Denoised stays within the oracle's parity bar."""
    full, only_den, eager = BenchFrames(), BenchFrames(), BenchFrames(eager=True)
    try:
        host_g = [{k: full.ctx.image_download(full.path.gsets[s][k]) for k in (HP.N_NORMALS, HP.N_MOTION)} for s in (0, 1)]
        state = O.SvgfState(W, H)
        for f in range(8):
            s, pfd = full.frame()
            only_den.frame()
            eager.frame()
            n0 = only_den.ctx.kernel_launches
            got = full.svgf_images()
            want = eager.svgf_images()
            den = only_den.denoised_async()
            assert only_den.ctx.kernel_launches == n0, "reading Denoised must not launch the pending last iteration"
            for k in want:
                assert np.array_equal(_bits(got[k]), _bits(want[k])), f"frame {f}: '{k}' differs from the immediate-launch run"
            assert np.array_equal(_bits(den), _bits(want["denoised"])), f"frame {f}: Denoised differs when only it is read back"
            rt = full.ctx.image_download(HP.N_RT)
            ref_den, _, _ = state.run(pfd, host_g[s][HP.N_NORMALS], host_g[s][HP.N_MOTION], rt, want_iters=False)
            Hh.assert_parity(got["denoised"], ref_den, f"frame {f} denoised vs oracle")
    finally:
        for b in (full, only_den, eager):
            b.close()


def test_last_iteration_costs_no_launch():
    """Steady-state frames launch one kernel fewer than the seven dispatches they issue (ray pass, svgf.comp, five a-trous)."""
    deferred, eager = BenchFrames(), BenchFrames(eager=True)
    try:
        for b in (deferred, eager):
            b.frame(); b.frame()
        n = 6
        counts = []
        for b in (deferred, eager):
            n0 = b.ctx.kernel_launches
            for _ in range(n):
                b.frame()
            counts.append(b.ctx.kernel_launches - n0)
        assert counts == [6 * n, 7 * n], counts
        assert np.array_equal(_bits(deferred.denoised_async()), _bits(eager.denoised_async()))
    finally:
        deferred.close(); eager.close()


class OneDispatch:
    """A context with noise in storage image `a`, normals bound, and step `step` of the filter dispatched a -> b (left pending)."""

    def __init__(self, normals, integ, pfd, eager=False, blit_alias=0, step=16):
        self.ctx = capi.Context(W, H)
        if eager:
            _eager(self.ctx)
        ctx = self.ctx
        ctx.set_option(capi.OPT_BLIT_ALIAS, blit_alias)
        ctx.update_per_frame_ubo(pfd)
        ctx.actualize_image(Hh.N_NORMALS, F4)
        ctx.actualize_image(Hh.N_DENOISED, F4)
        ctx.image_upload(Hh.N_NORMALS, normals)
        self.a, self.b, self.p = (ctx.upload_new_storage_image(W, H, F4) for _ in range(3))
        ctx.storage_image_upload(self.a, integ)
        ctx.bind_pass_images([Hh.N_NORMALS])
        self.pc = np.zeros((), T.SVGFPushConstants)
        self.pc["integrated_shadow_and_ao"] = (self.a, self.b)
        self.pc["atrous_step"] = step
        self.step = step

    def dispatch(self):
        self.ctx.dispatch(ATROUS, _groups(W), _groups(H), 1, self.pc)


@pytest.fixture(scope="module")
def inputs():
    _, _, frames = Hh.scene_and_gbuffer(W, H, moving=True)
    (pfd, g0), (_, g1) = frames[0], frames[2]
    assert not np.array_equal(_bits(g0["normals"]), _bits(g1["normals"]))
    return pfd, g0["normals"], g1["normals"], Hh.noise_integrated(H, W, seed=11)


def _eager_result(pfd, normals, integ):
    d = OneDispatch(normals, integ, pfd, eager=True)
    try:
        d.dispatch()
        return d.ctx.storage_image_download(d.b)
    finally:
        d.ctx.close()


def test_partial_upload_into_normals_launches_first(inputs):
    pfd, old, new, integ = inputs
    want = _eager_result(pfd, old, integ)
    d = OneDispatch(old, integ, pfd)
    try:
        d.dispatch()
        n0 = d.ctx.kernel_launches
        rows = np.ascontiguousarray(new[: H // 2])
        d.ctx.image_upload_rows_async(Hh.N_NORMALS, rows, 0, H // 2)
        assert d.ctx.kernel_launches == n0 + 1, "a write into the normals it reads must launch the pending dispatch first"
        got = d.ctx.storage_image_download(d.b)
        assert np.array_equal(_bits(got), _bits(want))
        Hh.assert_parity(got, O.svgf_atrous(pfd, old, integ, d.step), "pending dispatch vs oracle on the old normals")
        assert np.array_equal(_bits(d.ctx.image_download(Hh.N_NORMALS)[: H // 2]), _bits(rows))
    finally:
        d.ctx.close()


def test_full_upload_into_shared_normals_renames_and_keeps_the_dispatch_pending(inputs):
    """Normals shares its buffer with a storage image after a copy-free blit: a full upload takes a fresh buffer (make_writable), the
    dispatch keeps reading the old one and stays pending until its output is read."""
    pfd, old, new, integ = inputs
    want = _eager_result(pfd, old, integ)
    d = OneDispatch(old, integ, pfd, blit_alias=1)
    try:
        d.ctx.blit_transient_to_storage(Hh.N_NORMALS, d.p)
        d.dispatch()
        n0 = d.ctx.kernel_launches
        host = np.ascontiguousarray(new)
        d.ctx.image_upload_async(Hh.N_NORMALS, host)
        assert d.ctx.kernel_launches == n0, "a whole upload into a shared image renames it: nothing needs launching"
        got = d.ctx.storage_image_download(d.b)
        assert d.ctx.kernel_launches == n0 + 1
        assert np.array_equal(_bits(got), _bits(want))
        assert np.array_equal(_bits(d.ctx.storage_image_download(d.p)), _bits(old))
        assert np.array_equal(_bits(d.ctx.image_download(Hh.N_NORMALS)), _bits(new))
    finally:
        d.ctx.close()


def _driver():
    cu = C.CDLL("libcuda.so.1")
    cu.cuMemcpyDtoH_v2.argtypes = [C.c_void_p, C.c_uint64, C.c_size_t]
    return cu


def test_device_pointer_export_launches_first(inputs):
    pfd, old, _, integ = inputs
    want = _eager_result(pfd, old, integ)
    d = OneDispatch(old, integ, pfd)
    try:
        d.dispatch()
        n0 = d.ctx.kernel_launches
        ptr = d.ctx.storage_image_info(d.b)[0]
        assert d.ctx.kernel_launches == n0 + 1
        cu = _driver()
        assert cu.cuCtxSynchronize() == 0          # every stream of the device's context, not vhr_context_synchronize
        host = np.empty((H, W, 4), np.float16)
        assert cu.cuMemcpyDtoH_v2(host.ctypes.data, ptr, host.nbytes) == 0
        assert np.array_equal(_bits(host), _bits(want))
    finally:
        d.ctx.close()


@pytest.mark.parametrize("blit_alias", [0, 1])
def test_blit_source_launches_first(inputs, blit_alias):
    pfd, old, _, integ = inputs
    want = _eager_result(pfd, old, integ)
    d = OneDispatch(old, integ, pfd, blit_alias=blit_alias)
    try:
        d.dispatch()
        n0 = d.ctx.kernel_launches
        d.ctx.blit_storage_to_transient(d.b, Hh.N_DENOISED)
        assert d.ctx.kernel_launches == n0 + 1
        assert np.array_equal(_bits(d.ctx.image_download(Hh.N_DENOISED)), _bits(want))
    finally:
        d.ctx.close()


def test_whole_overwrite_drops_and_destroy_resolves(inputs):
    """The output overwritten whole before any read: never launched. Destroying the output image drops a pending dispatch; destroying
    an image it reads launches it first; destroying the context with one pending is clean, and the next context computes as before."""
    pfd, old, _, integ = inputs
    want = _eager_result(pfd, old, integ)
    d = OneDispatch(old, integ, pfd)
    try:
        d.dispatch()
        n0 = d.ctx.kernel_launches
        zeros = np.zeros((H, W, 4), np.float16)
        d.ctx.storage_image_upload(d.b, zeros)
        assert d.ctx.kernel_launches == n0, "an upload over the whole output drops the pending dispatch"
        assert np.array_equal(_bits(d.ctx.storage_image_download(d.b)), _bits(zeros))

        d.dispatch()
        capi._check(capi.lib().vhr_destroy_storage_image(d.ctx._h, d.b))
        assert d.ctx.kernel_launches == n0, "destroying the output drops the pending dispatch"

        c = d.ctx.upload_new_storage_image(W, H, F4)
        d.pc["integrated_shadow_and_ao"] = (d.a, c)
        d.dispatch()
        capi._check(capi.lib().vhr_destroy_transient_resources(d.ctx._h))
        assert d.ctx.kernel_launches == n0 + 1, "destroying the normals it reads launches it first"
        assert np.array_equal(_bits(d.ctx.storage_image_download(c)), _bits(want))

        d.ctx.actualize_image(Hh.N_NORMALS, F4)
        d.ctx.image_upload(Hh.N_NORMALS, old)
        d.ctx.bind_pass_images([Hh.N_NORMALS])
        d.dispatch()
    finally:
        d.ctx.close()                                   # one dispatch still pending
    assert _eager_result(pfd, old, integ).tobytes() == want.tobytes()
