"""python -m torch.distributed.run --nproc-per-node N tools/time_partition_gather.py [--parity-only] [--output-rank P] [--width W ...]

The gathered output of the fused partition (VHR_OPT_OUTPUT_RANK): the composition draw of every rank but P stores its band a second time
into rank P's RENDER_OUTPUT over NVLink, so rank P holds the whole frame. Workload: strong_4k's frame of bench.py (3840x2160, 3 M-triangle
sponza_like, shadow + 2 AO + reflection rays, 5-iteration SVGF), driven from the camera: partitioned G-Buffer Pass, Raytrace + SVGF, then the
composition (ray-traced shadows, AO and reflections) into a B8G8R8A8_SRGB RENDER_OUTPUT, alternating two camera poses.

--parity-only: every rank also renders the one-GPU frame in a context of its own; on the first --frames frames rank P's whole output is
compared with it bit for bit, and the run prints "PARITY OK (bit-exact)" (exit 0) or "PARITY FAILED" (exit 1).
Otherwise, after the same check, as the max over ranks of CUDA-event times, alternating the two settings in the same run:
  1. frame_gather_off / frame_gather_on   the N-GPU camera-in frame with the output rank off (-1) and on (P);
  2. draw_gather_off / draw_gather_on     the composition draw alone, off and on (on: the kernel and its two waits for all ranks).
With one rank only the one-GPU frame and its draw are measured; everything else is written as "not measured". Rank 0 writes the JSON
(--out) with the GPU's name and power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist

from vulkanhybridrenderer_b200 import camera, capi, scenes
from vulkanhybridrenderer_b200 import hybrid_path as HP
from vulkanhybridrenderer_b200 import multi_gpu as MG

LIGHT_DIR = (-0.3, -1.0, 0.2)        # bench.py's scene: seed 3, this light, two poses 5 cm / 0.002 rad apart
MODES = (HP.SHADOW_MODE_RAYTRACED, HP.AO_MODE_RAYTRACED, HP.REFLECTION_MODE_RAYTRACED)
FMT = HP.T.VK_FORMAT_B8G8R8A8_SRGB
NOT_MEASURED = "not measured (needs two or more GPUs)"


def power_limit_w(index):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return float(out)
    except Exception:
        return None


def compose(ctx, path, gset, rtset):
    g = path.gsets[gset]
    ctx.bind_pass_images([g[HP.N_ALBEDO], g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH], HP.N_SHADOW_MAP, HP.N_SSAO, HP.N_SSR,
                          HP.N_DENOISED, path.rt_sets[rtset][1], HP.N_RENDER_OUTPUT])
    ctx.draw(HP.SHADER_COMPOSITION, MODES)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--tris", type=int, default=3_000_000)
    ap.add_argument("--output-rank", type=int, default=0)
    ap.add_argument("--frames", type=int, default=4, help="frames of the parity check")
    ap.add_argument("--steps", type=int, default=30, help="timed frames (or draws) per repetition")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3, help="repetitions of each measurement, interleaved")
    ap.add_argument("--parity-only", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "time_partition_gather.json"))
    args = ap.parse_args()
    W, H = args.width, args.height
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    P = args.output_rank
    if not torch.cuda.is_available():
        raise SystemExit("time_partition_gather.py: no CUDA device")
    if world > 1 and not 0 <= P < world:
        raise SystemExit(f"time_partition_gather.py: --output-rank {P} is not a rank of {world}")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    sc = scenes.sponza_like(args.tris, seed=3, width=W, height=H)
    sc.light = camera.directional_light(LIGHT_DIR)
    cam = sc.camera
    poses = [(cam.position.copy(), cam.yaw, cam.pitch), (cam.position + np.array([0.05, 0.0, 0.01]), cam.yaw + 0.002, cam.pitch)]
    seq = camera.FrameSequencer(W, H, sc.light)
    pfds = [None, None]
    for s in (1, 0, 1):             # pose 1 first, so that each pose's previous camera is the other one
        cam.set_pose(*poses[s])
        pfds[s] = seq.next(cam)
    stream = torch.cuda.Stream()

    def make(**kw):
        ctx = capi.Context(W, H, device=local, stream=stream.cuda_stream)
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.set_option(capi.OPT_TRACE_SHADOWS, 1); ctx.set_option(capi.OPT_TRACE_AO, 1); ctx.set_option(capi.OPT_AO_SPP, 2)
        ctx.set_option(capi.OPT_TRACE_REFLECTIONS, 1)
        return ctx, HP.HybridRenderPath(ctx, W, H, gbuffer_sets=2, composition=FMT, shadow_map_size=(8, 8), **kw)

    def pfd_of(k):
        pfd = pfds[k & 1]
        pfd["frame_index"] = 3 + k
        return pfd

    def out_rows(c):
        p, w, h, f = c.image_info(HP.N_RENDER_OUTPUT)
        return torch.as_tensor(MG._DeviceRows(p, h, w * HP.T.FORMAT_TEXEL_BYTES[f] // 2), device="cuda")

    with torch.cuda.stream(stream):
        one, one_path = make(blit_alias=True)           # the best single-GPU configuration, as bench.py's strong_4k
        mv = 0.0                                        # motion halo of the two poses, from the single-GPU G-buffer
        for s in (0, 1):
            one.update_per_frame_ubo(pfds[s])
            one_path.gbuffer_pass(s)
            mv = max(mv, float(np.abs(one.image_download(one_path.gsets[s][HP.N_MOTION])[..., 1].astype(np.float32)).max()))
        motion_halo = min(64, MG.required_motion_halo(mv, H))
        one.close()
        one, one_path = make(blit_alias=True)           # fresh, like the partitioned context: the frames compared start alike

        def one_step(k):
            pfd = pfd_of(k)
            one.update_per_frame_ubo(pfd)
            one_path.gbuffer_pass(k & 1)
            one_path.frame(pfd, gset=k & 1)
            one_path.composition_pass(*MODES, denoised=True, gset=k & 1)

        result = {"tool": "tools/time_partition_gather.py", "n_gpus": world, "output_rank": P if world > 1 else None, "width": W, "height": H,
                  "triangles": int(sc.num_triangles), "render_output_format": "B8G8R8A8_SRGB", "rays_per_pixel": "1 shadow + 2 AO + 1 reflection",
                  "svgf_iterations": 5, "motion_halo_rows": motion_halo,
                  "gpu": torch.cuda.get_device_name(local), "power_limit_w": power_limit_w(local)}
        ok = True
        if world > 1:
            ctx, path = make(rt_sets=2)
            MG.setup_fused_partition(ctx, path, world, rank, motion_halo=motion_halo, exchange_gbuffer=True, output_rank=P)
            bands = [MG.band_rows(H, world, r)[0] for r in range(world)] + [H]

            def part_step(k):
                pfd = pfd_of(k)
                ctx.update_per_frame_ubo(pfd)
                path.gbuffer_pass(k & 1)
                path.frame(pfd, gset=k & 1, rtset=k & 1)
                compose(ctx, path, k & 1, k & 1)

            # ---- parity: rank P's whole output against its own one-GPU frame --------------------------------------------------------
            for k in range(args.frames):
                one_step(k)
                part_step(k)
                if rank == P:
                    bad = int((out_rows(ctx).view(torch.int16) != out_rows(one).view(torch.int16)).sum())
                    stream.synchronize()
                    print(f"[gather x{world}] frame {k}: output rank {P}: {bad} mismatching 16-bit words of {H * W * 2}", flush=True)
                    ok &= bad == 0
            flag = torch.tensor([0 if ok else 1], device="cuda")
            stream.synchronize()
            dist.broadcast(flag, P)
            ok = int(flag) == 0
            if rank == 0:
                print("[partition gather] PARITY", "OK (bit-exact)" if ok else "FAILED", flush=True)
        if not ok or args.parity_only:
            stream.synchronize()
            barrier()
            one.close()
            if world > 1:
                ctx.close()
                dist.destroy_process_group()
            sys.exit(0 if ok else 1)

        # ---- timing -----------------------------------------------------------------------------------------------------------
        frame_no = [args.frames]

        def timed(fn, n):
            """ms per call, max and min over ranks; every rank starts after a barrier"""
            for _ in range(args.warmup):
                fn(frame_no[0]); frame_no[0] += 1
            stream.synchronize()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(n):
                fn(frame_no[0]); frame_no[0] += 1
            e1.record(stream)
            e1.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / n], device="cuda", dtype=torch.float64)
            tmin = t.clone()
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            return float(t), float(tmin)

        def with_gather(on, fn):
            def run(k):
                ctx.set_option(capi.OPT_OUTPUT_RANK, P if on else -1)    # every rank switches at the same call of the same frame
                fn(k)
            return run

        arms = {"one_gpu_frame": one_step, "one_gpu_draw": lambda k: one_path.composition_pass(*MODES, denoised=True, gset=k & 1)}
        if world > 1:
            arms.update({"frame_gather_off": with_gather(False, part_step), "frame_gather_on": with_gather(True, part_step),
                         "draw_gather_off": with_gather(False, lambda k: compose(ctx, path, k & 1, k & 1)),
                         "draw_gather_on": with_gather(True, lambda k: compose(ctx, path, k & 1, k & 1))})
        times = {k: [] for k in arms}
        for _ in range(args.reps):
            for name, fn in arms.items():
                times[name].append(timed(fn, args.steps))
        stream.synchronize()
        barrier()

    def row(name, what):
        if name not in times:
            return {"ms": NOT_MEASURED, "what": what}
        mx = [t[0] for t in times[name]]
        return {"ms": float(np.median(mx)), "ms_reps_max_over_ranks": mx, "ms_reps_min_over_ranks": [t[1] for t in times[name]], "what": what}

    received = (H - (bands[P + 1] - bands[P])) * W * 4 if world > 1 else 0
    result.update({
        "steps": args.steps, "warmup": args.warmup, "reps": args.reps, "parity_frames": args.frames,
        "parity": f"bit-exact (rank {P}'s whole RENDER_OUTPUT against the one-GPU frame)" if world > 1 else "not checked (one rank)",
        "one_gpu_frame": row("one_gpu_frame", "one GPU: G-Buffer Pass + Raytrace + SVGF + composition, camera in (every rank at once, max over ranks)"),
        "one_gpu_draw": row("one_gpu_draw", "one GPU: the composition draw alone over the whole frame"),
        "frame_gather_off": row("frame_gather_off", "N GPUs: partitioned G-Buffer Pass + Raytrace + SVGF + composition, each rank keeps its band"),
        "frame_gather_on": row("frame_gather_on", "the same frame with the output rank on: the whole frame lands in its RENDER_OUTPUT"),
        "draw_gather_off": row("draw_gather_off", "N GPUs: the composition draw alone on the rank's band"),
        "draw_gather_on": row("draw_gather_on", "the composition draw alone with the output rank on: kernel + two waits for all ranks"),
        "bytes_received_by_output_rank_per_frame": received if world > 1 else NOT_MEASURED,
    })
    if world > 1:
        result["frame_cost_of_gather_ms"] = result["frame_gather_on"]["ms"] - result["frame_gather_off"]["ms"]
        result["draw_cost_of_gather_ms"] = result["draw_gather_on"]["ms"] - result["draw_gather_off"]["ms"]
    if rank == 0:
        print(json.dumps(result), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")
    one.close()
    if world > 1:
        ctx.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
