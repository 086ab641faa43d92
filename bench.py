#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native ray-traced lighting + SVGF chain.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one frame of the hybrid render path's hot chain on synthetic input:
    Raytrace Pass (shadow 1 spp + AO 1 spp per non-sky pixel)  ->  SVGF Denoise Pass (temporal + variance + 5 a-trous
    iterations, the reference's blits and ping-pong), 1920x1080, ~3M-triangle procedural scene (BASELINE.json north_star
    target configuration). The G-buffer (depth / normals+ids / motion) is an INPUT of the path.

metric  : shadow+AO Mrays/s over the whole frame (unique rays / frame time; the SVGF ms/frame and the ray pass' own
          Mrays/s ride along as extra keys). N > 1: every rank renders its own view of the replicated scene (BASELINE
          config 5 style, no data-path collective) => weak scaling; value = rays of all ranks / max-over-ranks time.
value   : inputs resident in HBM, CUDA-event timed.      e2e: same frames through the C-ABI with HOST G-buffers in
          pinned memory (H2D inside the timed region) and the denoised + raw shadow/AO images read back (D2H).
--impl reference : the CPU restatement of the reference shaders (oracle/, OpenMP on all host cores) on a bounded
          row-band sample of the same frame. The reference itself (Win32 + Vulkan + GLSL) cannot run here (DESIGN.md).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (width, height, triangles, ao_spp, reflections)
    "hybrid_frame_1080p_3Mtri": (1920, 1080, 3_000_000, 1, 0),       # north_star target (default)
    "shadows_1080p_260ktri": (1920, 1080, 260_000, 0, 0),            # BASELINE config 2
    "ao4_temporal_1080p_1Mtri": (1920, 1080, 1_000_000, 4, 0),       # BASELINE config 3
    "full_frame_4k_3Mtri": (3840, 2160, 3_000_000, 2, 1),            # BASELINE config 4 on one GPU (reference's 2 spp + reflections)
    "views64_1080p_3Mtri": (1920, 1080, 3_000_000, 2, 1),            # BASELINE config 5: 64 independent views, round-robin over the ranks (frames/s)
    "tiny": (320, 184, 20_000, 1, 0),                                # CPU-sized self-test of this script
}
SCENE_SEED = 3
LIGHT_DIR = (-0.3, -1.0, 0.2)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_scene(wl, view=0):
    from vulkanhybridrenderer_b200 import camera, scenes
    W, H, tris, _, _ = WORKLOADS[wl]
    sc = scenes.sponza_like(tris, seed=SCENE_SEED, width=W, height=H)
    sc.light = camera.directional_light(LIGHT_DIR)
    cam = sc.camera
    # two camera poses the bench oscillates between (non-trivial reprojection every frame); per-rank view offset
    base = cam.position + np.array([0.9 * view, 0.0, 0.0])
    poses = [(base, cam.yaw + 0.01 * view, cam.pitch), (base + np.array([0.05, 0.0, 0.01]), cam.yaw + 0.01 * view + 0.002, cam.pitch)]
    return sc, poses


class ClockSampler:
    """nvidia-smi style clock / throttle-reason samples taken DURING the timed region (pynvml, 10 ms period)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = str(e)

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._stop.set()
            self._thr.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement on a bounded row band (cpu_baseline of the default run and --impl reference)
# ---------------------------------------------------------------------------------------------------------------------
class CpuArm:
    def __init__(self, wl, band_rows):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_lib as O
        from vulkanhybridrenderer_b200 import camera
        self.O = O
        # all the host threads this process may use, set explicitly: torchrun exports OMP_NUM_THREADS=1 to every rank
        avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        self.cores = O.set_num_threads(avail)
        self.W, self.H, _, self.ao_spp, self.refl = WORKLOADS[wl]
        self.sc, self.poses = make_scene(wl)
        t0 = time.time()
        self.osc = O.OracleScene(self.sc)
        self.bvh_s = time.time() - t0
        self.seq = camera.FrameSequencer(self.W, self.H, self.sc.light)
        self.rows = min(band_rows, self.H)
        self.y0 = (self.H - self.rows) // 2
        # The SVGF pass (svgf.comp + five svgf_atrous_filter.comp dispatches, ~85 % of this arm's time) runs the REFERENCE'S OWN SHADERS compiled for
        # the CPU (oracle/_ref, built by oracle/make_ref.py where /root/reference exists; it travels to the GPU box as a built library) when that
        # library is there, else the hand-written port (bit-identical to it). The rays always go through the port's BVH: the reference's
        # traceRayEXT is the Vulkan driver, there is no reference CPU implementation of it.
        self.svgf_impl, self.kind = O, "port"
        try:
            import ref_lib
            if ref_lib.available():
                self.svgf_impl, self.kind = ref_lib, "reference"
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"bench.py: oracle/_ref not usable ({e}); the CPU arm runs the port\n")
        self.state = self.svgf_impl.SvgfState(self.W, self.rows)
        self.g = None
        self.k = 0

    def prepare(self):
        """G-buffer of the band for both camera poses (CPU primary rays; set-up, untimed)."""
        cam = self.sc.camera
        self.frames = []
        for pose in (self.poses[1], self.poses[0], self.poses[1]):
            cam.set_pose(*pose)
            pfd = self.seq.next(cam)
            self.frames.append((pfd, self.osc.gbuffer(pfd, self.W, self.H)))
        self.frames = self.frames[1:]

    def step(self):
        """One bounded sample: raygen on rows [y0, y0+rows) + the SVGF pass on that band. Returns (seconds, rays)."""
        pfd, g = self.frames[self.k & 1]
        pfd = pfd.copy()
        pfd["frame_index"] = 3 + self.k
        self.k += 1
        y0, y1 = self.y0, self.y0 + self.rows
        flags = 1 | (2 if self.ao_spp else 0) | (4 if self.refl else 0)
        t0 = time.perf_counter()
        out = self.osc.raygen(pfd, g["depth"], g["normals"], ao_spp=max(self.ao_spp, 1), flags=flags, rows=(y0, y1))
        t1 = time.perf_counter()
        band_pfd = pfd.copy()
        band_pfd["display_size"] = (self.W, self.rows)
        band_pfd["display_size_inverse"] = (np.float32(1) / np.float32(self.W), np.float32(1) / np.float32(self.rows))
        self.state.run(band_pfd, np.ascontiguousarray(g["normals"][y0:y1]), np.ascontiguousarray(g["motion"][y0:y1]),
                       np.ascontiguousarray(out["shadow_ao"][y0:y1]), want_iters=False)
        t2 = time.perf_counter()
        nonsky = int((g["depth"][y0:y1] > 0).sum())
        rays = nonsky * (1 + self.ao_spp + self.refl)
        return t2 - t0, rays, t1 - t0, t2 - t1

    def use_port_svgf(self):
        self.svgf_impl = self.O
        self.state = self.O.SvgfState(self.W, self.rows)

    def sample_desc(self):
        svgf = ("the reference's own svgf.comp + svgf_atrous_filter.comp compiled for the CPU (oracle/_ref)" if self.kind == "reference"
                else "the oracle port of the SVGF pass")
        return (f"a {self.rows}-ROW BAND, rows [{self.y0},{self.y0 + self.rows}) of the {self.W}x{self.H} frame (not a whole frame): ray generation + CPU BVH "
                f"traversal of the oracle port (shadow 1 + AO {self.ao_spp} spp{' + reflection' if self.refl else ''}; the reference's traceRayEXT is the "
                f"Vulkan driver) + {svgf} on that band, OpenMP {self.cores} threads")

    def full_frame_svgf_ms(self):
        """One actual full-frame SVGF pass of the oracle (the band figure extrapolates linearly; this one is measured)."""
        pfd, g = self.frames[0]
        st = self.svgf_impl.SvgfState(self.W, self.H)
        rt = np.zeros((self.H, self.W, 2), np.float16)
        rt[..., 0] = (np.arange(self.W)[None, :] // 7 + np.arange(self.H)[:, None] // 5) % 2
        rt[..., 1] = 0.5
        st.run(pfd, g["normals"], g["motion"], rt, want_iters=False)
        t0 = time.perf_counter()
        st.run(pfd, g["normals"], g["motion"], rt, want_iters=False)
        return (time.perf_counter() - t0) * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args.workload, args.cpu_rows)
    arm.prepare()
    for _ in range(args.warmup):
        arm.step()
    tot_s, tot_rays, rt_s, svgf_s = 0.0, 0, 0.0, 0.0
    for _ in range(args.steps):
        s, r, a, b = arm.step()
        tot_s += s; tot_rays += r; rt_s += a; svgf_s += b
    val = tot_rays / tot_s / 1e6
    W, H, tris, ao, refl = WORKLOADS[args.workload]
    full_svgf_ms = arm.full_frame_svgf_ms()
    port_val = val
    if arm.kind == "reference":          # the same steps with the port's SVGF pass (the faster, conservative CPU figure)
        arm.use_port_svgf()
        arm.step()
        ps, pr = 0.0, 0
        for _ in range(args.steps):
            s, r, _, _ = arm.step()
            ps += s; pr += r
        port_val = pr / ps / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "metric_note": f"CPU arm: each step is a {arm.rows}-ROW BAND of the frame, not a frame; the rate (rays / second) is scale-free",
        "value": val, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": tot_s / args.steps * 1e3, "ms_per_step_is": f"one {arm.rows}-row band, not a frame",
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**config_dict(args.workload, arm.sc.num_triangles), "frames_in_flight": args.frames_in_flight},
        "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": arm.cores, "kind": arm.kind, "sample": arm.sample_desc(), "port_value": port_val,
                         "raygen_s_per_step": rt_s / args.steps, "svgf_s_per_step": svgf_s / args.steps,
                         "svgf_ms_per_full_frame_extrapolated": svgf_s / args.steps * 1e3 * H / arm.rows,
                         "svgf_ms_per_full_frame_measured": full_svgf_ms},
        "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "SVGF pass (about 85 % of this arm's time): the reference's own svgf.comp / svgf_atrous_filter.comp compiled for the CPU (oracle/_ref, kind "
                "'reference') when that library is present, else the hand-written port, which is bit-identical to it and 1.7-3x faster (no glm temporaries, "
                "no generic image access) — cpu_baseline.port_value is the same sample with the port's SVGF pass, the conservative figure. The rays go through "
                "the port's ray generation and CPU BVH in both cases: raygen.rgen is hard-wired to 2 AO samples, a reflection ray and a 4x shadow loop, so "
                "it cannot run this configuration, and the reference's traceRayEXT is the Vulkan driver. The reference program itself needs Win32 + Vulkan "
                "ray tracing + glslang and cannot run here",
    }
    print(json.dumps(line))


FRAMES_IN_FLIGHT_DEFAULT = 1
METRIC = "shadow+AO Mrays/s (frame = RT shadow+AO pass + SVGF temporal + 5 a-trous)"


def config_dict(wl, n_tris):
    W, H, _, ao, refl = WORKLOADS[wl]
    return {"workload": wl, "width": W, "height": H, "triangles": int(n_tris), "shadow_spp": 1, "ao_spp": ao,
            "reflections": bool(refl), "svgf_atrous_iterations": 5,
            "l2_policy": "no explicit flush: the per-frame working set (BVH + triangle records + G-buffer + SVGF images) exceeds the 126 MB L2",
            "camera": "two poses alternating every frame (non-zero motion vectors), frame_index increments"}


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def pinned_bytes(torch, n, write_combined=False):
    """Pinned host buffer of n bytes as a uint8 tensor. write_combined: cudaHostAllocWriteCombined — an upload source the CPU only ever
    writes (by DMA at set-up); the PCIe reads then skip the snoop of the CPU caches."""
    if not write_combined:
        return torch.empty(n, dtype=torch.uint8, pin_memory=True)
    import ctypes as C
    rt = C.CDLL("libcudart.so.12")
    p = C.c_void_p()
    rc = rt.cudaHostAlloc(C.byref(p), C.c_size_t(n), C.c_uint(0x01 | 0x04))       # cudaHostAllocPortable | cudaHostAllocWriteCombined
    if rc != 0 or not p.value:
        return torch.empty(n, dtype=torch.uint8, pin_memory=True)
    return torch.frombuffer((C.c_ubyte * n).from_address(p.value), dtype=torch.uint8)        # lives until the process exits


def bind_rank_to_cores(world, local):
    """One slice of the visible CPUs per rank: the ranks' host threads (launch loop + copy submission) do not migrate onto each other."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        per = max(1, len(cpus) // max(world, 1))
        mine = cpus[local * per:(local + 1) * per]
        if mine:
            os.sched_setaffinity(0, mine)
        return len(mine)
    except (AttributeError, OSError):
        return None


def load_counters():
    """Per-launch ncu counters of the committed profile (profiles/kernel_counters.json): DRAM bytes and warp instructions."""
    for name in ("kernel_counters.json", "dram_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            with open(p) as f:
                d = json.load(f)
            return {k: (v if isinstance(v, dict) else {"dram_bytes": v}) for k, v in d.items()}
    return {}


class GpuFrameLoop:
    """One context + HybridRenderPath rendering the workload's frames: set-up (scene, BVH, G-buffers of the two alternating poses in HBM and
    in pinned host memory) and the step functions the measurements time."""

    def __init__(self, torch, wl, local, stream, view, svgf_mode, fif=1, host_copies=True):
        from vulkanhybridrenderer_b200 import camera, capi
        from vulkanhybridrenderer_b200 import hybrid_path as HP
        self.torch, self.capi, self.HP, self.stream, self.fif = torch, capi, HP, stream, fif
        self.W, self.H, _, self.ao_spp, self.refl = WORKLOADS[wl]
        W, H = self.W, self.H
        self.sc, self.poses = make_scene(wl, view=view)
        ctx = self.ctx = capi.Context(W, H, device=local, stream=stream.cuda_stream)
        ctx.update_geometry(self.sc.vertices, self.sc.indices, self.sc.primitives)
        self.bvh = ctx.bvh_stats()
        ctx.set_option(capi.OPT_TRACE_SHADOWS, 1)
        ctx.set_option(capi.OPT_TRACE_AO, 1 if self.ao_spp else 0)
        ctx.set_option(capi.OPT_AO_SPP, max(self.ao_spp, 1))
        ctx.set_option(capi.OPT_TRACE_REFLECTIONS, self.refl)
        self.path = HP.HybridRenderPath(ctx, W, H, gbuffer_sets=2, rt_sets=2 if fif == 2 else 1, svgf_fused=svgf_mode == "fused",
                                        blit_alias=svgf_mode != "reference")
        self.seq = camera.FrameSequencer(W, H, self.sc.light)
        self.cam = self.sc.camera
        self.pfds, self.host_g, nonsky = [None, None], [None, None], []
        for s in (1, 0, 1):           # pose 1 first so that pose 0's "previous camera" is pose 1 and vice versa
            self.cam.set_pose(*self.poses[s])
            pfd = self.seq.next(self.cam)
            self.gbuffer_pass(pfd, s)
            self.pfds[s] = pfd
        for s in (0, 1):
            g, hg = self.path.gsets[s], {}
            for key in (HP.N_DEPTH, HP.N_NORMALS, HP.N_MOTION):
                _, w, h, f = ctx.image_info(g[key])
                t = pinned_bytes(torch, h * w * HP.T.FORMAT_TEXEL_BYTES[f])
                ctx.image_download_into(g[key], t)
                hg[key] = t
            ctx.synchronize()
            nonsky.append(int((hg[HP.N_DEPTH].view(torch.float32) > 0).sum()))
            if host_copies:       # the upload sources: write-combined copies of the same bytes
                for key in list(hg):
                    wc = pinned_bytes(torch, hg[key].numel(), write_combined=True)
                    wc.copy_(hg[key])
                    hg[key] = wc
            self.host_g[s] = hg
        self.rays_per_frame = [n * (1 + self.ao_spp + self.refl) for n in nonsky]
        self.h2d_bytes = sum(t.numel() for t in self.host_g[0].values())
        self.frame_no = 0

    def gbuffer_pass(self, pfd, s):
        HP, g = self.HP, self.path.gsets[s]
        self.ctx.update_per_frame_ubo(pfd)
        with self.ctx.debug_label("G-Buffer Pass"):
            self.ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
            self.ctx.gbuffer_pass(self.W, self.H)

    def next_pfd(self):
        k = self.frame_no
        s = k & 1
        pfd = self.pfds[s]
        pfd["frame_index"] = 3 + k
        self.frame_no += 1
        return k, s, pfd

    def step(self, overlap=True):
        k, s, pfd = self.next_pfd()
        if self.fif == 2 and overlap:
            self.path.frame_overlapped(pfd, k, gset=s)
        else:
            self.path.frame(pfd, gset=s, rtset=s if self.fif == 2 else 0)
        return self.rays_per_frame[s]

    def step_camera_in(self):
        """The path driven from a CAMERA: the per-frame constants (584 B) are the only input that crosses PCIe; the G-buffer producer pass
        (primary rays on the same BVH, SURVEY 8f rank 2) runs inside the step."""
        k, s, pfd = self.next_pfd()
        self.gbuffer_pass(pfd, s)
        self.path.frame(pfd, gset=s, rtset=0)
        return self.rays_per_frame[s]

    def upload_async(self, k):
        g = self.path.gsets[k & 1]
        for key, t in self.host_g[k & 1].items():
            self.ctx.image_upload_async(g[key], t)

    def close(self):
        self.ctx.close()


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, loop, rank, world):
    """--dump-outputs: what the last timed step handed its caller, as float32 .npy files: the denoised shadow/AO image, the raw ray-traced
    shadow/AO masks and, with reflections on, the reflection image ([H, W, C] each). Above the 64 MB budget (4K frames, or several ranks)
    every array keeps the same seeded sample of pixels ([n, C], pixel indices ascending), so two builds can still be compared value for value."""
    HP = loop.HP
    k = loop.frame_no - 1
    rt, refl = loop.path.rt_sets[(k & 1) if loop.fif == 2 else 0]
    images = {"denoised_shadow_ao": HP.N_DENOISED, "raytraced_shadow_ao": rt}
    if loop.refl:
        images["raytraced_reflections"] = refl
    arrays = {name: loop.ctx.image_download(img).astype(np.float32) for name, img in images.items()}
    px = loop.W * loop.H
    per_px = sum(a.nbytes for a in arrays.values()) // px
    if per_px * px * world > DUMP_BUDGET_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(px, DUMP_BUDGET_BYTES // (per_px * world), replace=False))
        arrays = {name: a.reshape(px, -1)[idx] for name, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + (f"_rank{rank}" if world > 1 else "") + ".npy"), a)


def timed(torch, stream, barrier, fn, n):
    """n calls of fn between two CUDA events on `stream`, barrier + synchronize on both sides. Returns (ms, sum of fn's return values)."""
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    tot = 0
    for _ in range(n):
        tot += fn()
    e1.record(stream)
    barrier()
    return e0.elapsed_time(e1), tot


def measure_e2e(torch, loop, barrier, K, Wm):
    """End to end through the C-ABI from HOST buffers, every step: 41.5 MB (1080p) of G-buffer up from pinned memory, the denoised image
    down. serial = blocking copies around the frame; pipelined (headline) = the same copies on the transfer queues, step k+1's upload
    and step k-1's read-back under step k's kernels, the host waiting for the previous read-back every step; camera_in = the per-frame
    constants are the only upload, the G-buffer producer pass runs inside the step."""
    ctx, HP, W, H, stream = loop.ctx, loop.HP, loop.W, loop.H, loop.stream
    capi = loop.capi
    out_den = pinned_bytes(torch, W * H * 8)
    d2h = out_den.numel()

    def step_serial():
        g = loop.path.gsets[loop.frame_no & 1]
        for key, t in loop.host_g[loop.frame_no & 1].items():
            capi._check(capi.lib().vhr_image_upload(ctx._h, g[key].encode(), t.data_ptr(), t.numel()))
        r = loop.step(overlap=False)
        ctx.image_download_into(HP.N_DENOISED, out_den)
        ctx.synchronize()
        return r

    for _ in range(max(2, Wm // 2)):
        step_serial()
    serial_ms, rays_serial = timed(torch, stream, barrier, step_serial, K)
    checksum_serial = float(out_den.view(torch.float16)[::4097].float().nan_to_num().sum())

    outs = [pinned_bytes(torch, W * H * 8) for _ in range(2)]

    def run_pipelined(n, step_fn, upload):
        rays_p, prev = 0, None
        if upload:
            loop.upload_async(loop.frame_no)
        for i in range(n):
            if upload:
                loop.upload_async(loop.frame_no + 1)        # next step's inputs (the last one primes the following run)
            rays_p += step_fn()
            t1 = ctx.image_download_async(HP.N_DENOISED, outs[i & 1])
            if prev is not None:
                ctx.wait_download(prev)
            prev = t1
        ctx.wait_download(prev)
        return rays_p

    res = {}
    for name, step_fn, upload in (("pipelined", lambda: loop.step(overlap=False), True), ("camera_in", loop.step_camera_in, False)):
        run_pipelined(max(3, Wm // 2), step_fn, upload)
        ctx.synchronize()
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        rays_e = run_pipelined(K, step_fn, upload)
        e1.record(stream)          # the host has already waited for the last read-back: this stamps its completion
        ctx.synchronize()
        barrier()
        res[name] = {"ms": max(e0.elapsed_time(e1), 0.0), "wall_ms": (time.perf_counter() - t0) * 1e3, "rays": rays_e,
                     "checksum": float(outs[(K - 1) & 1].view(torch.float16)[::4097].float().nan_to_num().sum())}
    res["serial"] = {"ms": serial_ms, "rays": rays_serial, "checksum": checksum_serial}
    res["d2h"] = d2h
    return res


def measure_next_rows(torch, loop):
    """SURVEY 8f rows, each timed on its own and NOT part of the step."""
    ctx, HP, W, H, stream, path, capi = loop.ctx, loop.HP, loop.W, loop.H, loop.stream, loop.path, loop.capi
    next_ms = {}
    try:
        path_c = HP.HybridRenderPath.__new__(HP.HybridRenderPath)
        path_c.ctx, path_c.W, path_c.H, path_c.gsets = ctx, W, H, path.gsets
        path_c.ssao_radius = np.array(0.75, np.float32)
        path_c.ssr_pc = np.array((25.0, 0.1, 0.5, 10), HP.T.SSRPushConstants)
        for n, f in ((HP.N_SSAO_RAW, HP.F4), (HP.N_SSAO, HP.F4), (HP.N_SSR, HP.F4)):
            ctx.actualize_image(n, f)
        ctx.actualize_image(HP.N_SHADOW_MAP, HP.T.VK_FORMAT_D32_SFLOAT, 4096, 4096)
        ctx.actualize_image(HP.N_RENDER_OUTPUT, HP.T.VK_FORMAT_B8G8R8A8_SRGB)
        row_reps = int(os.environ.get("VHR_BENCH_ROW_REPS", "0"))      # profiling runs: a few launches per row are enough

        def time_row(fn, reps=20):
            reps = row_reps or reps
            ctx.update_per_frame_ubo(loop.pfds[0])
            for _ in range(3):
                fn(0)
            ec0, ec1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ec0.record(stream)
            for i in range(reps):
                fn(i & 1)
            ec1.record(stream)
            torch.cuda.synchronize()
            return ec0.elapsed_time(ec1) / reps

        def ssao_only(s):
            g = path.gsets[s]
            ctx.bind_pass_images([g[HP.N_NORMALS], g[HP.N_DEPTH], HP.N_SSAO_RAW])
            ctx.dispatch(HP.SHADER_SSAO, HP.groups(W), HP.groups(H), 1, path_c.ssao_radius)

        def blur_only(s):
            ctx.bind_pass_images([HP.N_SSAO_RAW, HP.N_SSAO])
            ctx.dispatch(HP.SHADER_SSAO_BLUR, HP.groups(W), HP.groups(H), 1, path_c.ssao_radius)

        def gbuffer_only(s):
            g = path.gsets[s]
            ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
            ctx.gbuffer_pass(W, H)

        next_ms["composition"] = time_row(lambda s: path_c.composition_pass(0, 0, 0 if loop.refl else 2, denoised=True, gset=s))
        next_ms["ssao"] = time_row(ssao_only)
        next_ms["ssao_blur"] = time_row(blur_only)
        next_ms["ssr"] = time_row(lambda s: path_c.ssr_pass(gset=s), reps=6)
        # the producer rewrites the resident G-buffer of pose 0 with identical values (same camera, same scene)
        next_ms["gbuffer"] = time_row(lambda s: gbuffer_only(0), reps=6)
    except capi.VhrError as e:      # never let the extra rows break the headline measurement
        sys.stderr.write(f"bench.py: next rows skipped: {e}\n")
    return next_ms


def measure_strong_4k(torch, dist, args, local, rank, world, stream, barrier):
    """BASELINE config 4 / north_star's multi-GPU claim: ONE 3840x2160 frame (shadow + 2 AO + reflection rays per pixel, 5-iteration SVGF,
    3 M triangles) over the N GPUs of the box: fused partition (ray pass in 8-row blocks dealt round-robin with the results stored into the
    owners' images over NVLink peer memory, SVGF on row bands with halo rows pushed by the kernels, flag words; no collective in the frame).
    The one-GPU time of the SAME frame is measured first, on every rank at once (max over ranks), so the speed-up is self-contained."""
    from vulkanhybridrenderer_b200 import capi
    from vulkanhybridrenderer_b200 import hybrid_path as HP
    from vulkanhybridrenderer_b200 import multi_gpu as MG
    wl = "full_frame_4k_3Mtri"
    W, H, _, ao_spp, refl = WORKLOADS[wl]
    K1, K2, Wm = 8, max(10, min(args.steps, 30)), 3
    # ---- one GPU: the unpartitioned frame, best single-GPU configuration --------------------------------------------------------------
    one = GpuFrameLoop(torch, wl, local, stream, 0, "alias", host_copies=False)
    for _ in range(Wm):
        one.step()
    ms1, _ = timed(torch, stream, barrier, one.step, K1)
    host_g, rays_frame, pfds, n_tris = one.host_g, one.rays_per_frame, one.pfds, one.sc.num_triangles
    one.close()
    # ---- N GPUs ----------------------------------------------------------------------------------------------------------------------
    sc, poses = make_scene(wl, view=0)
    y0, y1 = MG.band_rows(H, world, rank)
    ctx = capi.Context(W, H, device=local, stream=stream.cuda_stream)
    ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
    ctx.set_option(capi.OPT_TRACE_AO, 1); ctx.set_option(capi.OPT_AO_SPP, ao_spp); ctx.set_option(capi.OPT_TRACE_REFLECTIONS, refl)
    path = HP.HybridRenderPath(ctx, W, H, gbuffer_sets=2, rt_sets=2)
    for s in (0, 1):       # full G-buffer of both poses into HBM (set-up, untimed), from the host copies of the one-GPU run
        for key, t in host_g[s].items():
            capi._check(capi.lib().vhr_image_upload(ctx._h, path.gsets[s][key].encode(), t.data_ptr(), t.numel()))
    mv = max(float(host_g[s][HP.N_MOTION].view(torch.float16).view(H, W, 4)[..., 1].float().abs().max()) for s in (0, 1))
    motion_halo = min(64, MG.required_motion_halo(mv, H))
    MG.setup_fused_partition(ctx, path, world, rank, motion_halo=motion_halo)
    frame_no = [0]

    def step():
        k = frame_no[0]; s = k & 1
        pfd = pfds[s]; pfd["frame_index"] = 3 + k
        frame_no[0] += 1
        path.frame(pfd, gset=s, rtset=k & 1)          # the plain single-GPU call sequence
        return 0

    for _ in range(Wm):
        step()
    l0 = ctx.kernel_launches
    msN, _ = timed(torch, stream, barrier, step, K2)
    launches = ctx.kernel_launches - l0
    # ---- e2e: every step this rank uploads the G-buffer rows it consumes and reads its band of the results back -----------------------
    #   depth + normals of the 8-row blocks it ray-traces (one strided DMA each), normals + motion of its SVGF band +- halo rows;
    #   down: its band of the denoised image and of the reflections. Pipelined on the transfer queues like the 1-GPU e2e.
    blocks = [b for b in range((H + 7) // 8) if b % world == rank and b * 8 + 8 <= H]
    # normals: the a-trous taps of the widest iteration reach 32 rows beyond the band, and the band's copy into the previous-frame normals is
    # read up to motion_halo + 1 rows beyond it by the next temporal pass; motion vectors are only read at the pixel itself
    halo = max(32, motion_halo + 1) + 8
    n0, n1 = max(0, y0 - halo), min(H, y1 + halo)
    row = {HP.N_DEPTH: W * 4, HP.N_NORMALS: W * 8, HP.N_MOTION: W * 8}
    outs = [(pinned_bytes(torch, (y1 - y0) * W * 8), pinned_bytes(torch, (y1 - y0) * W * 8)) for _ in range(2)]
    h2d = len(blocks) * 8 * (row[HP.N_DEPTH] + row[HP.N_NORMALS]) + (n1 - n0) * row[HP.N_NORMALS] + (y1 - y0) * row[HP.N_MOTION]
    d2h = 2 * (y1 - y0) * W * 8

    def upload(k):
        s = k & 1
        g = path.gsets[s]
        if blocks:
            for key in (HP.N_DEPTH, HP.N_NORMALS):
                ctx.image_upload_blocks_async(g[key], host_g[s][key], blocks[0] * 8, 8, world * 8, len(blocks))
        ctx.image_upload_rows_async(g[HP.N_NORMALS], host_g[s][HP.N_NORMALS][n0 * row[HP.N_NORMALS]:], n0, n1)
        ctx.image_upload_rows_async(g[HP.N_MOTION], host_g[s][HP.N_MOTION][y0 * row[HP.N_MOTION]:], y0, y1)

    def run_e2e(n):
        prev = None
        upload(frame_no[0])
        for i in range(n):
            upload(frame_no[0] + 1)
            k = frame_no[0]
            step()
            o = outs[i & 1]
            t1 = ctx.image_download_rows_async(HP.N_DENOISED, o[0], y0, y1)
            t2 = ctx.image_download_rows_async(path.rt_sets[k & 1][1], o[1], y0, y1)
            if prev is not None:
                ctx.wait_download(prev)
            prev = max(t1, t2)
        ctx.wait_download(prev)
        return 0

    run_e2e(3)
    ctx.synchronize()
    msE, _ = timed(torch, stream, barrier, lambda: run_e2e(K2), 1)
    den = torch.as_tensor(MG._DeviceRows(ctx.image_info(HP.N_DENOISED)[0], H, W * 4), device="cuda")
    band_sum = den[y0:y1].float().nan_to_num().sum().double()
    t = torch.tensor([ms1 / K1, msN / K2, msE / K2], device="cuda", dtype=torch.float64)
    tmax, tmin = t.clone(), t.clone()
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
    r = torch.tensor([float(band_sum), float(launches), float(h2d), float(d2h)], device="cuda", dtype=torch.float64)
    dist.all_reduce(r, op=dist.ReduceOp.SUM)
    ctx.close()
    rays = float(np.mean(rays_frame))
    ms1f, msNf, msEf = (float(x) for x in tmax.cpu())
    return {
        "workload": wl, "scaling": "strong", "n_gpus": world, "width": W, "height": H, "triangles": int(n_tris), "rays_per_frame": rays,
        "partition": "fused: ray pass in 8-row blocks dealt round-robin, results stored into the owners' images over NVLink peer memory; SVGF on row "
                     "bands, halo rows pushed by the kernels; stream-ordered flag words; no collective in the frame",
        "motion_halo_rows": motion_halo,
        "ms_per_frame_1gpu": ms1f, "ms_per_frame": msNf, "speedup_vs_1gpu": ms1f / msNf, "efficiency": ms1f / msNf / world,
        "mrays_s_1gpu": rays / ms1f / 1e3, "mrays_s": rays / msNf / 1e3,
        "ms_per_frame_min_over_ranks": float(tmin.cpu()[1]), "frames_timed": K2, "gpu_launches_all_ranks": int(r[1]),
        "e2e": {"ms_per_frame": msEf, "mrays_s": rays / msEf / 1e3, "speedup_vs_1gpu_device_time": ms1f / msEf,
                "h2d_bytes_per_step_all_ranks": int(r[2]), "d2h_bytes_per_step_all_ranks": int(r[3]),
                "what": "per rank and step: depth + normals of its ray blocks (strided DMA), normals of its band +- (a-trous / motion halo) rows and motion "
                        "vectors of its band up; its band of the denoised image and of the reflections down; copies on the transfer queues under the kernels"},
        "denoised_checksum": float(r[0]),
    }


def run_views64(args):
    """BASELINE config 5 as specified: a batch of 64 independent camera views of the ~3 M-triangle scene (seeded ring of cameras), BVH replicated,
    view v -> rank v mod N, no collective. Every view is a whole frame from a CAMERA: G-buffer producer pass (primary rays), Raytrace Pass with the
    reference's ray set (1 shadow + 2 AO + 1 reflection ray per pixel), SVGF Denoise Pass; the denoised image of every view is read back."""
    import torch
    import torch.distributed as dist
    from vulkanhybridrenderer_b200 import camera, capi
    from vulkanhybridrenderer_b200 import hybrid_path as HP
    from vulkanhybridrenderer_b200 import multi_gpu as MG
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        bind_rank_to_cores(world, local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W, H, tris, ao_spp, refl = WORKLOADS[args.workload]
    n_views = 64
    stream = torch.cuda.Stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        from vulkanhybridrenderer_b200 import scenes
        sc = scenes.sponza_like(tris, seed=SCENE_SEED, width=W, height=H)
        sc.light = camera.directional_light(LIGHT_DIR)
        ctx = capi.Context(W, H, device=local, stream=stream.cuda_stream)
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.set_option(capi.OPT_AO_SPP, ao_spp); ctx.set_option(capi.OPT_TRACE_REFLECTIONS, refl)
        path = HP.HybridRenderPath(ctx, W, H, svgf_fused=False, blit_alias=True)
        cam = sc.camera
        base, yaw0 = cam.position.copy(), cam.yaw
        rng = np.random.default_rng(64)
        ring = [(base + np.array([0.9 * np.cos(2 * np.pi * v / n_views), 0.15 * rng.uniform(-1, 1), 0.9 * np.sin(2 * np.pi * v / n_views)]),
                 yaw0 + 2 * np.pi * v / n_views, cam.pitch) for v in range(n_views)]
        mine = MG.views_for_rank(n_views, world, rank)
        pfds = []
        for v in mine:
            cam.set_pose(*ring[v])
            pfds.append(camera.FrameSequencer(W, H, sc.light, first_frame_index=3 + v).next(cam))      # an independent frame: previous camera = this camera
        outs = [pinned_bytes(torch, W * H * 8) for _ in range(2)]
        g = path.gsets[0]
        rays_of = {}

        def batch():
            prev, n = None, 0
            for i, pfd in enumerate(pfds):
                ctx.update_per_frame_ubo(pfd)
                with ctx.debug_label("G-Buffer Pass"):
                    ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
                    ctx.gbuffer_pass(W, H)
                path.frame(pfd)
                t = ctx.image_download_async(HP.N_DENOISED, outs[i & 1])
                if prev is not None:
                    ctx.wait_download(prev)
                prev = t
                n += 1
            ctx.wait_download(prev)
            return n

        batch()       # warm-up batch; also counts the rays of every view once
        for i, pfd in enumerate(pfds):
            ctx.update_per_frame_ubo(pfd)
            ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
            ctx.gbuffer_pass(W, H)
            rays_of[i] = int((ctx.image_download(g[HP.N_DEPTH]) > 0).sum()) * (1 + ao_spp + refl)
        reps = args.steps // n_views
        sampler = ClockSampler(local)
        l0 = ctx.kernel_launches
        barrier(); sampler.start()
        ms, frames = timed(torch, stream, barrier, batch, reps)
        clocks = sampler.stop()
        launches = ctx.kernel_launches - l0
        rays = sum(rays_of.values()) * reps
        ctx.close()
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t)
        r = torch.tensor([frames, rays, launches], device="cuda", dtype=torch.float64); dist.all_reduce(r, op=dist.ReduceOp.SUM)
        frames, rays, launches = (float(x) for x in r.cpu())
    if rank == 0:
        print(json.dumps({
            "metric": "frames/s over a batch of 64 independent 1080p views (camera in, denoised image out)", "value": frames / (ms * 1e-3), "unit": "frames/s",
            "n_gpus": world, "steps": int(frames), "warmup": n_views, "ms_per_step": ms / (frames / world), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "views": n_views, "width": W, "height": H, "triangles": int(sc.num_triangles), "shadow_spp": 1, "ao_spp": ao_spp,
                       "reflections": bool(refl), "svgf_atrous_iterations": 5, "partition": "view v -> rank v mod N, BVH replicated, no collective",
                       "per_view": "G-buffer producer pass + Raytrace Pass + SVGF Denoise Pass; 584 B of per-frame constants up, 16.6 MB denoised image down"},
            "mrays_s": rays / (ms * 1e-3) / 1e6, "ms_per_view": ms / (frames / world), "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": frames / (ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": 584, "d2h_bytes_per_step": W * H * 8}}))
    if world > 1:
        dist.destroy_process_group()


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from vulkanhybridrenderer_b200 import hybrid_path as HP

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    cores = bind_rank_to_cores(world, local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    wl = args.workload
    W, H, _, ao_spp, refl = WORKLOADS[wl]
    fif = args.frames_in_flight
    # queue 0 carries the short SVGF kernels: with two frames in flight it gets the higher priority so that its CTAs are placed as
    # the long ray kernel's CTAs retire instead of queueing behind that kernel's whole grid
    stream = torch.cuda.Stream(priority=-1) if fif == 2 else torch.cuda.Stream()
    K, Wm = args.steps, args.warmup
    peak, peak_src = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        loop = GpuFrameLoop(torch, wl, local, stream, rank, args.svgf, fif)
        ctx, path, sc, st = loop.ctx, loop.path, loop.sc, loop.bvh

        # ---- value: inputs resident in HBM ----------------------------------------------------------------------------
        path.timestamps = None
        for _ in range(Wm):
            loop.step()
        if fif == 1:
            path.enable_timestamps(K)
        l0 = ctx.kernel_launches
        sampler = ClockSampler(local)
        barrier()
        sampler.start()
        ms_total, rays = timed(torch, stream, barrier, loop.step, K)
        clocks = sampler.stop()
        launches = ctx.kernel_launches - l0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, loop, rank, world)
        if fif == 2:
            # per-pass times need the passes one after the other: the same frames again, one frame in flight, with timestamps
            Kb = min(K, 50)
            path.enable_timestamps(Kb)
            for _ in range(Kb):
                loop.step(overlap=False)
            barrier()
            pass_ms = path.pass_times_ms(Kb)
        else:
            pass_ms = path.pass_times_ms(K)            # [K, passes]
        path.timestamps = None

        next_ms = measure_next_rows(torch, loop) if world == 1 or rank == 0 else {}
        barrier()
        e2e = measure_e2e(torch, loop, barrier, K, Wm)
        h2d = loop.h2d_bytes
        loop.close()
        strong = measure_strong_4k(torch, dist, args, local, rank, world, stream, barrier) if world > 1 and not args.no_strong else None

    # ---- reduce over ranks: max time, summed rays ------------------------------------------------------------------------
    e2e_ms, e2e_wall_ms, e2e_serial_ms, cam_ms = e2e["pipelined"]["ms"], e2e["pipelined"]["wall_ms"], e2e["serial"]["ms"], e2e["camera_in"]["ms"]
    rays_e, rays_serial, rays_cam = e2e["pipelined"]["rays"], e2e["serial"]["rays"], e2e["camera_in"]["rays"]
    if world > 1:
        t = torch.tensor([ms_total, e2e_ms, e2e_wall_ms, e2e_serial_ms, cam_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_ms, e2e_wall_ms, e2e_serial_ms, cam_ms = (float(x) for x in t.cpu())
        r = torch.tensor([rays, rays_e, launches, rays_serial, rays_cam], device="cuda", dtype=torch.float64)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
        rays, rays_e, launches, rays_serial, rays_cam = (float(x) for x in r.cpu())

    if rank == 0:
        px = W * H
        mean_pass = pass_ms.mean(axis=0)
        labels = path.PASS_LABELS
        pm = dict(zip(labels, (float(x) for x in mean_pass)))
        frame_ms = ms_total / K
        svgf_ms = sum(pm[k] for k in labels if k != "raytrace")
        # shares are taken of the frame run one pass after the other (with two frames in flight the passes overlap and their
        # durations no longer add up to the step)
        share_ms = sum(pm.values()) if fif == 2 else frame_ms
        counters = load_counters()
        sm_clock_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        # per-kernel roofline (HBM): algorithmic bytes / launch = per-pixel bytes (DESIGN.md) x pixels; plus, where the committed ncu profile has
        # the kernel's warp-instruction count, the fraction of the machine's issue slots (148 SMs x 4 schedulers x SM clock) the launch used
        kernels = []

        def add(name, ms, bytes_, note=None):
            ach = bytes_ / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            k = {"kernel": name, "ms": ms, "share": ms / share_ms, "algorithmic_bytes": bytes_, "achieved_gbs": ach, "frac": ach / peak}
            c = counters.get(name.split(" ")[0], {})
            if c.get("inst_executed") and ms > 0:
                k["issue"] = {"warp_instructions_per_launch": c["inst_executed"], "achieved_ginst_s": c["inst_executed"] / (ms * 1e-3) / 1e9,
                              "peak_ginst_s": 148 * 4 * sm_clock_hz / 1e9, "frac": c["inst_executed"] / (ms * 1e-3) / (148 * 4 * sm_clock_hz),
                              "source": "instruction count from the committed ncu profile (profiles/kernel_counters.json), duration live"}
            if note:
                k["note"] = note
            kernels.append(k)
        add("raygen_kernel", pm["raytrace"], px * (HP.BYTES_RAYGEN_IO + (8 if refl else 0)),
            "traversal-bound (software BVH, no RT cores): compulsory G-buffer in + mask out bytes only; see Mrays/s and issue.frac")
        fused = args.svgf == "fused"
        add("svgf_fused_kernel (svgf.comp + a-trous iteration 0)" if fused else "svgf_temporal_kernel", pm["svgf_temporal"],
            px * (HP.BYTES_TEMPORAL + (8 if fused else 0)))
        at_ms = float(np.mean([pm[f"atrous{i}"] for i in (1, 2, 3, 4)]))
        add("atrous_pair_kernel (mean of iterations 1-4)", at_ms, px * HP.BYTES_ATROUS)
        if not fused:
            add("atrous_pair_kernel (iteration 0, + the history blit of the reference sequence)", pm["atrous0"],
                px * (HP.BYTES_ATROUS + (HP.BYTES_BLIT if args.svgf == "reference" else 0)))
        add("blits (prev-normals, denoised)" + ("" if args.svgf == "reference" else ": copy-on-write aliases, no copy"), pm["blits"],
            px * 2 * HP.BYTES_BLIT if args.svgf == "reference" else 0)
        dom = max(kernels[:3], key=lambda k: k["ms"])
        cdom = counters.get(dom["kernel"].split(" ")[0], {})
        roofline = {"kernel": dom["kernel"], "bound": "hbm", "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": dom["frac"], "traffic": cdom.get("dram_bytes"), "peak_source": peak_src, "ms_per_launch": dom["ms"],
                    "share_of_step": dom["share"]}
        if "issue" in dom:
            roofline["issue"] = dom["issue"]
        if dom["kernel"] == "raygen_kernel":
            # the contract's roofline is HBM or tensor; a software BVH traversal is bound by neither — say what does bound it
            roofline["note"] = ("not an HBM-bound kernel: software BVH traversal (no RT cores on B200) bound by instruction issue and node-fetch latency "
                                "at ~15 of 32 lanes active per instruction (ncu, profiles/), DRAM at 2 % of peak; the figures of merit are "
                                "rt_pass.mrays_s and roofline.issue.frac. The HBM-bound part of the step is the SVGF chain: svgf.frac_of_peak_vs_fused_minimum")
        svgf_bytes = px * (HP.BYTES_TEMPORAL + 5 * HP.BYTES_ATROUS + 3 * HP.BYTES_BLIT)
        svgf_min_bytes = px * 148
        line = {
            "metric": METRIC, "value": rays / (ms_total * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": frame_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {**config_dict(wl, sc.num_triangles), "frames_in_flight": fif, "svgf_mode": args.svgf,
                       **({"multi_gpu": "one independent view of the replicated scene per rank, no data-path collective (BASELINE config 5 style); the "
                                        "strong-scaling 4K row-band frame of config 4 is measured in the same run: key strong_4k",
                           "host_cores_per_rank": cores} if world > 1 else {}),
                       **({"schedule": "Raytrace Pass of frame k+1 on queue 1 under the SVGF pass of frame k (two ray-output image sets); "
                                       "kernels[] / roofline timed in a separate run with one frame in flight",
                           "ms_per_step_one_frame_in_flight": share_ms} if fif == 2 else {})},
            "e2e": {"value": rays_e / (e2e_ms * 1e-3) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": e2e["d2h"],
                    "ms_per_step": e2e_ms / K, "wall_ms_per_step": e2e_wall_ms / K, "checksum": e2e["pipelined"]["checksum"],
                    "mode": "pipelined: G-buffer (depth, normals, motion) up from write-combined pinned memory and the denoised image down on the C-ABI "
                            "transfer queues, copies of consecutive steps under the kernels, host waits for step k-1's read-back during step k",
                    "serial_ms_per_step": e2e_serial_ms / K, "serial_value": rays_serial / (e2e_serial_ms * 1e-3) / 1e6,
                    "serial_checksum": e2e["serial"]["checksum"],
                    "host_device_gbs_all_ranks": (h2d + e2e["d2h"]) * world / (e2e_ms / K * 1e-3) / 1e9,
                    **({"limiter": "N > 1: every rank moves its own 58 MB per step; the box's host<->device fabric (all GPUs on one NUMA node of a 32-vCPU "
                                   "host) delivered 109 / 119 / 153 GB/s in aggregate at 2 / 4 / 8 GPUs (profiles/r02_summary.md), i.e. 54 / 30 / 19 GB/s per GPU: the "
                                   "G-buffer-in rate stops scaling there, the camera-in rate (no G-buffer over PCIe) and the device rate do not"} if world > 1 else {}),
                    "camera_in": {"value": rays_cam / (cam_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": cam_ms / K, "h2d_bytes_per_step": 584,
                                  "d2h_bytes_per_step": e2e["d2h"], "checksum": e2e["camera_in"]["checksum"],
                                  "what": "the path driven from a camera: only the per-frame constants go up, the G-buffer producer pass (primary rays, "
                                          "SURVEY 8f rank 2) runs inside the step, the denoised image comes down"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "kernels": kernels,
            "rt_pass": {"ms": pm["raytrace"], "mrays_s": (rays / K / world) / (pm["raytrace"] * 1e-3) / 1e6, "rays_per_frame": rays / K / world},
            "svgf": {"ms_per_frame": svgf_ms, "reference_dataflow_bytes": svgf_bytes, "achieved_gbs": svgf_bytes / (svgf_ms * 1e-3) / 1e9,
                     "frac_of_peak": svgf_bytes / (svgf_ms * 1e-3) / 1e9 / peak,
                     "fused_minimum_bytes": svgf_min_bytes, "frac_of_peak_vs_fused_minimum": svgf_min_bytes / (svgf_ms * 1e-3) / 1e9 / peak},
            "bvh": {"triangles": st.n_triangles, "wide_nodes": st.n_wide_nodes, "build_ms": st.build_ms, "sah_cost": st.sah_cost},
        }
        if strong:
            line["strong_4k"] = strong
        if next_ms:
            rows = {"composition": ("composition_kernel", px * (HP.BYTES_COMPOSITION + (8 if refl else 0)), None),
                    "ssao": ("ssao_kernel", px * HP.BYTES_SSAO, "depth quad-image pre-pass + 16 samples per pixel in the oracle's operations (the sample position must be exact: the filter "
                             "coordinate is quantised to 1/256 texel; the occlusion term cancels eight digits next to the pixel): issue-bound (89 %), "
                             "the depth gather at 47 % of the L1"),
                    "ssao_blur": ("ssao_blur_kernel", px * HP.BYTES_SSAO_BLUR, None),
                    "ssr": ("ssr_kernel", px * HP.BYTES_SSR, "up to 250 march steps + 10 bisection steps per pixel, each one re-projection + bilinear depth tap in the oracle's "
                            "operations (the two comparisons decided from a bounded estimate): instruction-bound, the HBM fraction is tiny by construction"),
                    "gbuffer": ("gbuffer_kernel", px * 28, "primary closest-hit rays on the BVH (traversal-bound); 28 B/px of G-buffer written")}
            line["next_rows"] = {}
            for key, ms_ in next_ms.items():
                kname, b_, note = rows[key]
                line["next_rows"][key] = {"kernel": kname, "ms": ms_, "algorithmic_bytes": b_, "achieved_gbs": b_ / (ms_ * 1e-3) / 1e9,
                                          "frac": b_ / (ms_ * 1e-3) / 1e9 / peak, "note": (note + "; " if note else "") + "timed on its own after the frames, not part of the step"}
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(wl, args.cpu_rows)
            arm.prepare()
            arm.step()
            t_s, t_r, n = 0.0, 0, 0
            svgf_s = 0.0
            while n < 3 or (t_s < 8.0 and n < 10):
                s_, r_, _, b_ = arm.step()
                t_s += s_; t_r += r_; svgf_s += b_; n += 1
            line["cpu_baseline"] = {"value": t_r / t_s / 1e6, "unit": "Mrays/s", "cores": arm.cores, "kind": arm.kind,
                                    "sample": arm.sample_desc() + f", {n} samples",
                                    "svgf_ms_per_full_frame_extrapolated": svgf_s / n * 1e3 * H / arm.rows,
                                    "svgf_ms_per_full_frame_measured": arm.full_frame_svgf_ms()}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm, row-band partition of ONE frame (BASELINE config 4): strong scaling, NCCL halo exchange per a-trous iteration
# ---------------------------------------------------------------------------------------------------------------------
def run_rowband(args):
    import torch
    import torch.distributed as dist
    from vulkanhybridrenderer_b200 import camera, capi
    from vulkanhybridrenderer_b200 import hybrid_path as HP
    from vulkanhybridrenderer_b200 import multi_gpu as MG

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = args.workload
    W, H, _, ao_spp, refl = WORKLOADS[wl]
    sc, poses = make_scene(wl, view=0)          # every rank renders the SAME view; the scene and BVH are replicated
    fif = args.frames_in_flight
    # queue 0 carries the short SVGF kernels: with two frames in flight it gets the higher priority so that its CTAs are placed as
    # the long ray kernel's CTAs retire instead of queueing behind that kernel's whole grid
    stream = torch.cuda.Stream(priority=-1) if fif == 2 else torch.cuda.Stream()
    K, Wm = args.steps, args.warmup
    y0, y1 = MG.band_rows(H, world, rank)
    with torch.cuda.stream(stream):
        ctx = capi.Context(W, H, device=local, stream=stream.cuda_stream)
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.set_option(capi.OPT_TRACE_AO, 1 if ao_spp else 0)
        ctx.set_option(capi.OPT_AO_SPP, max(ao_spp, 1))
        ctx.set_option(capi.OPT_TRACE_REFLECTIONS, refl)
        fused = args.halo == "fused" and world > 1
        path = HP.HybridRenderPath(ctx, W, H, gbuffer_sets=2, rt_sets=2 if fused else 1)
        seq = camera.FrameSequencer(W, H, sc.light)
        cam = sc.camera
        pfds = [None, None]
        # G-buffer input (untimed set-up). NCCL mode: band + halo rows. Fused mode: the ray pass is interleaved over the
        # whole frame, so every rank is given the full G-buffer.
        g0, g1 = (0, H) if fused else (max(0, y0 - MG.GBUFFER_HALO), min(H, y1 + MG.GBUFFER_HALO))
        ctx.set_option(capi.OPT_ROW_BEGIN, g0); ctx.set_option(capi.OPT_ROW_END, g1)
        for s_ in (1, 0, 1):
            cam.set_pose(*poses[s_])
            pfd = seq.next(cam)
            ctx.update_per_frame_ubo(pfd)
            g = path.gsets[s_]
            ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH]])
            ctx.gbuffer_pass(W, H)
            pfds[s_] = pfd
        nonsky = [int((ctx.image_download(path.gsets[s_][HP.N_DEPTH])[y0:y1] > 0).sum()) for s_ in (0, 1)]
        frame_no = [0]
        if args.motion_halo <= 0:       # auto: what this camera motion needs (every rank sees the same G-buffer rows it compares)
            mv = max(float(np.abs(ctx.image_download(path.gsets[s_][HP.N_MOTION])[g0:g1, :, 1].astype(np.float32)).max()) for s_ in (0, 1))
            t = torch.tensor([mv], device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            args.motion_halo = min(64, MG.required_motion_halo(float(t), H))
        if fused:
            MG.setup_fused_partition(ctx, path, world, rank, motion_halo=args.motion_halo)
            drivers = []

            def step():
                k = frame_no[0]; s_ = k & 1
                pfd = pfds[s_]; pfd["frame_index"] = 3 + k
                frame_no[0] += 1
                path.frame(pfd, gset=s_, rtset=k & 1)          # the plain single-GPU call sequence
                return nonsky[s_] * (1 + ao_spp + refl)
        else:
            backends = [MG.CabiBandBackend(ctx, path, gset=s_) for s_ in (0, 1)]
            drivers = [MG.RowBandSvgf(b, H, world, rank, motion_halo=args.motion_halo) for b in backends]

            def step():
                k = frame_no[0]; s_ = k & 1
                pfd = pfds[s_]; pfd["frame_index"] = 3 + k
                frame_no[0] += 1
                ctx.update_per_frame_ubo(pfd)
                backends[s_].trace((y0, y1))
                drivers[s_].run()
                return nonsky[s_] * (1 + ao_spp + refl)

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        for _ in range(Wm):
            step()
        l0 = ctx.kernel_launches
        sampler = ClockSampler(local)
        barrier(); sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        rays = 0
        for _ in range(K):
            rays += step()
        ev1.record(stream)
        barrier()
        clocks = sampler.stop()
        ms_total = ev0.elapsed_time(ev1)
        launches = ctx.kernel_launches - l0
        sent = sum(d.x.bytes_sent for d in drivers) / max(1, frame_no[0])
        # stitched result for the checksum / parity (outside the timed region)
        den = torch.as_tensor(MG._DeviceRows(ctx.image_info(HP.N_DENOISED)[0], H, W * 4), device="cuda")
        band_sum = den[y0:y1].float().nan_to_num().sum().double()
    if world > 1:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms_total = float(t)
        r = torch.tensor([rays, launches, float(band_sum), sent], device="cuda", dtype=torch.float64); dist.all_reduce(r, op=dist.ReduceOp.SUM)
        rays, launches, band_sum, sent = (float(x) for x in r.cpu())
    if rank == 0:
        cfg = config_dict(wl, sc.num_triangles)
        how = ("ray pass in 8-row blocks dealt round-robin with results stored into the owners' images over NVLink peer memory, SVGF on row bands "
               "with halo rows pushed by the kernels, stream-ordered flag words; no collective in the frame") if args.halo == "fused" and world > 1 else \
              "NCCL halo exchange (6 grouped send/recv per frame), ray pass on the contiguous band"
        cfg.update({"partition": f"row bands x{world}, BVH replicated, {how}", "motion_halo_rows": args.motion_halo})
        print(json.dumps({
            "metric": METRIC, "value": rays / (ms_total * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "gpu_launches": int(launches), "clocks": clocks, "halo_bytes_per_frame_all_ranks": sent,
            "denoised_checksum": float(band_sum)}))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="hybrid_frame_1080p_3Mtri", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-rows", type=int, default=64, help="rows of the frame the CPU arm renders per sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--frames-in-flight", type=int, default=FRAMES_IN_FLIGHT_DEFAULT, choices=[1, 2],
                    help="2: the Raytrace Pass of frame k+1 is recorded on the context's second queue and runs under the SVGF pass of frame k "
                         "(HybridRenderPath.frame_overlapped); the per-kernel breakdown then comes from a separate one-frame-at-a-time run")
    ap.add_argument("--svgf", default="alias", choices=["reference", "alias", "fused"],
                    help="how the library answers the SVGF node's (unchanged) call sequence: reference = temporal kernel, five a-trous kernels, three "
                         "copies; alias = the three blits alias buffers copy-on-write (VHR_OPT_BLIT_ALIAS); fused = alias + svgf.comp and a-trous "
                         "iteration 0 in one kernel (VHR_OPT_SVGF_FUSED). Same images in all three (tests/test_svgf_gpu.py)")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the strong-scaling 4K frame (key strong_4k)")
    ap.add_argument("--partition", default="views", choices=["views", "rows"],
                    help="N>1: independent views per rank (weak scaling, default) or row bands of one frame (strong scaling, NCCL halos)")
    ap.add_argument("--halo", default="fused", choices=["fused", "nccl"],
                    help="row-band mode: halo rows pushed by the kernels over NVLink peer memory (default) or NCCL send/recv between passes")
    ap.add_argument("--motion-halo", type=int, default=0,
                    help="rows of history/moments exchanged for the temporal pass (row-band mode); 0 = derive from the G-buffer's motion vectors")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the images the last one computed to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload.startswith("views64") and args.steps % 64:
        ap.error("--workload views64_*: a step is one view and the views are timed in whole batches of 64, so --steps must be a multiple of 64")
    if args.dump_outputs and (args.impl == "reference" or args.workload.startswith("views64") or args.partition == "rows"):
        ap.error("--dump-outputs applies to the GPU frame loop (--impl b200, one view per rank)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload.startswith("views64"):
        run_views64(args)
    elif args.partition == "rows":
        run_rowband(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
