"""python -m torch.distributed.run --nproc-per-node N tools/time_partition_camera_in.py [--parity-only] [--width W --height H --tris T ...]

The fused partition driven from a CAMERA: the G-Buffer Pass runs partitioned (every rank traces the 8-row blocks its ray pass traces
and stores them into every rank's G-buffer over NVLink), then the plain single-GPU frame (Raytrace + SVGF) runs on the partition.
Default workload: strong_4k's frame of bench.py (3840x2160, 3 M-triangle sponza_like, shadow + 2 AO + reflection rays, 5-iteration
SVGF), alternating two camera poses and two G-buffer sets.

First, on the first --frames frames, every rank's band of the denoised image and of the reflections is compared with rank 0's
single-GPU frame bit for bit; any difference exits non-zero. Then, as the max over ranks of CUDA-event times:
  1. one_gpu_camera_in      the one-GPU camera-in frame (G-Buffer Pass + Raytrace + SVGF), run on every rank at once;
  2. replicated_producer    the N-GPU frame with the whole G-Buffer Pass on every rank (partition off, full pass, partition on);
  3. partitioned_producer   the N-GPU frame with the partitioned G-Buffer Pass;
  4. gbuffer_pass           the partitioned G-Buffer Pass on its own (its two waits included) against the unpartitioned one.
With one rank only 1 and the unpartitioned pass are measured. Rank 0 writes the JSON (--out) with the GPU's name and power limit."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--tris", type=int, default=3_000_000)
    ap.add_argument("--frames", type=int, default=4, help="frames of the parity check")
    ap.add_argument("--steps", type=int, default=30, help="timed frames per repetition")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3, help="repetitions of each measurement, interleaved")
    ap.add_argument("--parity-only", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "time_partition_camera_in.json"))
    args = ap.parse_args()
    W, H = args.width, args.height
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("time_partition_camera_in.py: no CUDA device")
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
        return ctx, HP.HybridRenderPath(ctx, W, H, gbuffer_sets=2, **kw)

    def pfd_of(k):
        pfd = pfds[k & 1]
        pfd["frame_index"] = 3 + k
        return pfd

    with torch.cuda.stream(stream):
        one, one_path = make(blit_alias=True)           # the best single-GPU configuration, as bench.py's strong_4k
        # motion halo of the two poses, from the single-GPU G-buffer
        mv = 0.0
        for s in (0, 1):
            one.update_per_frame_ubo(pfds[s])
            one_path.gbuffer_pass(s)
            mv = max(mv, float(np.abs(one.image_download(one_path.gsets[s][HP.N_MOTION])[..., 1].astype(np.float32)).max()))
        motion_halo = min(64, MG.required_motion_halo(mv, H))
        one.close()
        one, one_path = make(blit_alias=True)

        def one_step(k):
            pfd = pfd_of(k)
            one.update_per_frame_ubo(pfd)
            one_path.gbuffer_pass(k & 1)
            one_path.frame(pfd, gset=k & 1)

        result = {"tool": "tools/time_partition_camera_in.py", "n_gpus": world, "width": W, "height": H, "triangles": int(sc.num_triangles),
                  "rays_per_pixel": "1 shadow + 2 AO + 1 reflection", "svgf_iterations": 5, "motion_halo_rows": motion_halo,
                  "gpu": torch.cuda.get_device_name(local), "power_limit_w": power_limit_w(local)}
        ok = True
        if world > 1:
            ctx, path = make(rt_sets=2)
            MG.setup_fused_partition(ctx, path, world, rank, motion_halo=motion_halo, exchange_gbuffer=True)
            bands = [MG.band_rows(H, world, r)[0] for r in range(world)] + [H]
            y0, y1 = bands[rank], bands[rank + 1]

            def part_step(k):
                pfd = pfd_of(k)
                ctx.update_per_frame_ubo(pfd)
                path.gbuffer_pass(k & 1)
                path.frame(pfd, gset=k & 1, rtset=k & 1)

            def replicated_step(k):
                pfd = pfd_of(k)
                ctx.clear_partition()
                ctx.update_per_frame_ubo(pfd)
                path.gbuffer_pass(k & 1)
                ctx.set_partition(world, rank, bands, ray_block_rows=8, motion_halo=motion_halo)
                path.frame(pfd, gset=k & 1, rtset=k & 1)

            def rows(c, name):
                p, w, h, f = c.image_info(name)
                return torch.as_tensor(MG._DeviceRows(p, h, w * HP.T.FORMAT_TEXEL_BYTES[f] // 2), device="cuda")

            # ---- parity: fresh contexts, same frames ------------------------------------------------------------------------------
            for k in range(args.frames):
                one_step(k)
                part_step(k)
                bad_total = []
                for key, mine_name, ref_name in (("denoised", HP.N_DENOISED, HP.N_DENOISED), ("reflections", path.rt_sets[k & 1][1], HP.N_REFL)):
                    mine = rows(ctx, mine_name)[y0:y1].contiguous()
                    parts = [torch.empty((bands[r + 1] - bands[r], mine.shape[1]), dtype=mine.dtype, device="cuda") for r in range(world)]
                    stream.synchronize()
                    dist.all_gather(parts, mine)
                    if rank == 0:
                        got = torch.cat(parts).view(torch.int16)
                        want = rows(one, ref_name).view(torch.int16)
                        stream.synchronize()
                        bad = int((got != want).sum())
                        bad_total.append(f"{key} {bad}")
                        ok &= bad == 0
                if rank == 0:
                    print(f"[camera-in x{world}] frame {k}: mismatching halfs: " + ", ".join(bad_total), flush=True)
            flag = torch.tensor([0 if ok else 1], device="cuda")
            dist.broadcast(flag, 0)
            ok = int(flag) == 0
            if rank == 0:
                print("[camera-in partition] PARITY", "OK (bit-exact)" if ok else "FAILED", flush=True)
        if not ok or args.parity_only:
            stream.synchronize()
            barrier()
            if world > 1:
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

        def one_gbuffer(k):
            one.update_per_frame_ubo(pfd_of(k))
            one_path.gbuffer_pass(k & 1)

        def part_gbuffer(k):
            ctx.update_per_frame_ubo(pfd_of(k))
            path.gbuffer_pass(k & 1)

        arms = {"one_gpu_camera_in": one_step, "one_gpu_gbuffer_pass": one_gbuffer}
        if world > 1:
            arms.update({"replicated_producer": replicated_step, "partitioned_producer": part_step, "partitioned_gbuffer_pass": part_gbuffer})
        times = {k: [] for k in arms}
        for _ in range(args.reps):
            for name, fn in arms.items():
                times[name].append(timed(fn, args.steps))
        stream.synchronize()
        barrier()

    def row(name, what):
        if name not in times:
            return {"ms": "not measured", "what": what}
        mx = [t[0] for t in times[name]]
        return {"ms": float(np.median(mx)), "ms_reps_max_over_ranks": mx, "ms_reps_min_over_ranks": [t[1] for t in times[name]], "what": what}

    dealt_rows = [min(8, H - b * 8) for b in range((H + 7) // 8) if b % world == rank] if world > 1 else []
    peer_bytes = torch.tensor([28.0 * W * sum(dealt_rows) * (world - 1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(peer_bytes, op=dist.ReduceOp.MAX)
    result.update({
        "steps": args.steps, "warmup": args.warmup, "reps": args.reps, "parity_frames": args.frames,
        "parity": "bit-exact (denoised + reflections, every band)" if world > 1 else "not checked (one rank)",
        "one_gpu_camera_in": row("one_gpu_camera_in", "one GPU: G-Buffer Pass + Raytrace + SVGF, camera in (every rank at once, max over ranks)"),
        "replicated_producer": row("replicated_producer", "N GPUs: whole G-Buffer Pass on every rank (partition off, full pass, partition on) + partitioned frame"),
        "partitioned_producer": row("partitioned_producer", "N GPUs: partitioned G-Buffer Pass (rows dealt as the ray pass deals them, stored to every rank) + partitioned frame"),
        "gbuffer_pass": {"partitioned": row("partitioned_gbuffer_pass", "partitioned G-Buffer Pass alone, two alternating sets: kernel + trailing wait for all ranks"),
                         "unpartitioned": row("one_gpu_gbuffer_pass", "the single-GPU G-Buffer Pass over the whole frame")},
        "peer_store_bytes_per_rank_and_frame": float(peer_bytes) if world > 1 else 0.0,
    })
    if world > 1:
        result["speedup_partitioned_vs_replicated"] = result["replicated_producer"]["ms"] / result["partitioned_producer"]["ms"]
        result["speedup_partitioned_vs_one_gpu"] = result["one_gpu_camera_in"]["ms"] / result["partitioned_producer"]["ms"]
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
