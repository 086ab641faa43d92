"""python -m torch.distributed.run --nproc-per-node N tools/time_partition_shadow_map.py [--parity-only] [--tris 260000,3000000 ...]

The Shadow Map Pass under the fused partition: every rank rasterises the 8-row blocks of the 4096^2 map dealt to it (block b to rank
b % N) and stores them into every rank's map over NVLink, against the replicated pass (every rank renders the whole map).

First every rank's partitioned map is compared with its own replicated map bit for bit (both windows, then a zero light), and the
per-rank differences are summed over the ranks; any difference exits non-zero. Then, with CUDA events around --iters passes after
--warmup passes, repetitions interleaved, times per rank (max and min over ranks):
  1. shadow_map              the replicated and the partitioned pass, sponza_like at each --tris, reference and fitted window;
  2. zero_light_pass         the partitioned pass with a zero projview: both waits, the clear of the rank's rows and the push;
  3. push_kernel             shadow_push_kernel alone (torch.profiler, CUDA activities, in a run of its own after the timings);
  4. frame_4k                the 3840 x 2160 camera-in rasterised-shadow frame (G-Buffer Pass, Shadow Map Pass, SSAO, composition)
                             at --tris' largest, on one GPU (every rank at once) against the N-GPU partition.
With one rank only the replicated pass and the one-GPU frame are measured; the rest is recorded as not measured. Rank 0 writes the
JSON (--out) with the GPU's name and power limit, read in the same run."""
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
from vulkanhybridrenderer_b200 import types as T

S = 4096
D32 = T.VK_FORMAT_D32_SFLOAT
NOT_MEASURED = "not measured"
MODES = (HP.SHADOW_MODE_RASTERIZED, HP.AO_MODE_SSAO, HP.REFLECTION_MODE_OFF)


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return float(out)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tris", default="260000,3000000", help="sponza_like triangle counts")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3, help="repetitions of each measurement, interleaved")
    ap.add_argument("--frame-steps", type=int, default=30, help="timed frames of the 4K frame per repetition")
    ap.add_argument("--parity-only", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "time_partition_shadow_map.json"))
    args = ap.parse_args()
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("time_partition_shadow_map.py: no CUDA device")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    stream = torch.cuda.Stream()
    dw, dh = 64, 64 * max(world, 1)                  # display extent of the map-only contexts: the least the bands allow
    bands_small = [MG.band_rows(dh, world, r)[0] for r in range(world)] + [dh]

    def reduce(x, op):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=op)
        return float(t)

    def map_context(sc):
        """a context with the scene and a 4096^2 map, the map attached for every other rank over CUDA IPC"""
        ctx = capi.Context(dw, dh, device=local, stream=stream.cuda_stream)
        ctx.update_geometry(sc.vertices, sc.indices, sc.primitives)
        ctx.actualize_image(HP.N_SHADOW_MAP, D32, S, S)
        if world > 1:
            mine = (ctx.sync_export_ipc(), ctx.image_export_ipc(HP.N_SHADOW_MAP))
            everyone = [None] * world
            ctx.synchronize()
            dist.all_gather_object(everyone, mine)
            for r, (h_sync, h_map) in enumerate(everyone):
                if r != rank:
                    ctx.sync_attach_peer(r, h_sync)
                    ctx.image_attach_peer(HP.N_SHADOW_MAP, r, h_map)
            barrier()
        return ctx

    def set_light(ctx, sc, pv):
        light = sc.light.copy()
        light["projview"] = pv
        ctx.update_per_frame_ubo(camera.FrameSequencer(dw, dh, light).next(sc.camera))

    def map_pass(ctx, partitioned):
        if partitioned:
            ctx.set_partition(world, rank, bands_small)
        else:
            ctx.clear_partition()
        ctx.bind_pass_images([HP.N_SHADOW_MAP])
        ctx.shadow_map_pass()

    def timed(fn, n, warmup):
        """ms per call, (max, min) over ranks; every rank starts after a barrier"""
        for _ in range(warmup):
            fn()
        stream.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1) / n
        return reduce(ms, dist.ReduceOp.MAX), reduce(ms, dist.ReduceOp.MIN)

    def summary(reps, what):
        if not reps:
            return {"ms": NOT_MEASURED, "what": what}
        return {"ms_max_over_ranks": float(np.median([t[0] for t in reps])), "ms_min_over_ranks": float(np.median([t[1] for t in reps])),
                "reps": [list(t) for t in reps], "what": what}

    result = {"tool": "tools/time_partition_shadow_map.py", "n_gpus": world, "map": f"{S}x{S} D32_SFLOAT",
              "gpu": torch.cuda.get_device_name(local), "power_limit_w": power_limit_w(local),
              "iters": args.iters, "warmup": args.warmup, "reps": args.reps, "runs": []}
    ok = True
    tri_counts = [int(x) for x in args.tris.split(",")]
    with torch.cuda.stream(stream):
        # ---- parity and per-pass timings, per scene ----------------------------------------------------------------------------
        for n in tri_counts:
            sc = scenes.sponza_like(n, seed=3)
            ctx = map_context(sc)
            d = sc.light["direction"][:3]
            lo, hi = np.array(ctx.bvh_stats().scene_min), np.array(ctx.bvh_stats().scene_max)
            windows = {"reference": camera.light_projview(d), "fitted": camera.fit_light_projview(d, lo, hi)}
            row = {"triangles": int(ctx.bvh_stats().n_triangles)}
            if world > 1:
                for name, pv in list(windows.items()) + [("zero", np.zeros((4, 4), np.float32))]:
                    set_light(ctx, sc, pv)
                    map_pass(ctx, False)
                    want = ctx.image_download(HP.N_SHADOW_MAP)
                    map_pass(ctx, True)
                    got = ctx.image_download(HP.N_SHADOW_MAP)
                    bad = reduce(int(np.sum(got.view(np.uint32) != want.view(np.uint32))), dist.ReduceOp.SUM)
                    if rank == 0:
                        print(f"[partition shadow map x{world}] {row['triangles']} triangles, {name} window: {int(bad)} mismatching texels "
                              f"over all ranks ({np.mean(want > 0) * 100:.1f}% covered)", flush=True)
                    ok &= bad == 0
            if args.parity_only or not ok:
                stream.synchronize()
                barrier()
                ctx.close()
                continue
            for name, pv in windows.items():
                set_light(ctx, sc, pv)
                arms = {"replicated": lambda: map_pass(ctx, False)}
                if world > 1:
                    arms["partitioned"] = lambda: map_pass(ctx, True)
                reps = {k: [] for k in arms}
                for _ in range(args.reps):
                    for k, fn in arms.items():
                        reps[k].append(timed(fn, args.iters, args.warmup))
                row[f"{name}_window"] = {
                    "replicated": summary(reps["replicated"], "whole map on every rank"),
                    "partitioned": summary(reps.get("partitioned"), "rank's 8-row blocks, pushed to every rank; both waits included")}
                if rank == 0:
                    print(f"[partition shadow map x{world}] {row['triangles']} triangles, {name}: {json.dumps(row[f'{name}_window'])}", flush=True)
            zero = []
            if world > 1:
                set_light(ctx, sc, np.zeros((4, 4), np.float32))
                for _ in range(args.reps):
                    zero.append(timed(lambda: map_pass(ctx, True), args.iters, args.warmup))
            row["zero_light_pass"] = summary(zero, "partitioned pass with a zero projview: two waits, clear of the rank's rows, push")
            result["runs"].append(row)
            stream.synchronize()
            barrier()                                # the peers' last pushes into this map have landed before it is freed
            ctx.close()
        if world > 1:
            flag = torch.tensor([0 if ok else 1], device="cuda")
            dist.broadcast(flag, 0)
            ok = int(flag) == 0
            if rank == 0:
                print("[partition shadow map] PARITY", "OK (bit-exact)" if ok else "FAILED", flush=True)
        if not ok or args.parity_only:
            stream.synchronize()
            barrier()
            if world > 1:
                dist.destroy_process_group()
            sys.exit(0 if ok else 1)

        # ---- the 4K camera-in rasterised-shadow frame ------------------------------------------------------------------------------
        W, H = 3840, 2160
        sc = scenes.sponza_like(max(tri_counts), seed=3, width=W, height=H)
        fctx = capi.Context(W, H, device=local, stream=stream.cuda_stream)
        fctx.load_scene(sc)
        path = HP.HybridRenderPath(fctx, W, H, ssao=True, composition=T.VK_FORMAT_B8G8R8A8_SRGB, shadow_map_size=(S, S))
        pfd = camera.FrameSequencer(W, H, sc.light).next(sc.camera)
        fctx.update_per_frame_ubo(pfd)
        bands = None
        if world > 1:
            bands = MG.setup_fused_partition(fctx, path, world, rank, exchange_gbuffer=True, exchange_shadow_map=True)

        def frame(partitioned):
            if world > 1:
                if partitioned:
                    fctx.set_partition(world, rank, bands)
                else:
                    fctx.clear_partition()
            path.gbuffer_pass()
            path.shadow_map_pass()
            path.ssao_passes()
            path.composition_pass(*MODES)

        arms = {"one_gpu": lambda: frame(False)}
        if world > 1:
            arms["partitioned"] = lambda: frame(True)
        reps = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, fn in arms.items():
                reps[k].append(timed(fn, args.frame_steps, 3))
        result["frame_4k"] = {
            "width": W, "height": H, "triangles": int(fctx.bvh_stats().n_triangles),
            "passes": "G-Buffer Pass, Shadow Map Pass (4096^2, reference window), SSAO + blur, composition (rasterised shadows, SSAO, no reflections)",
            "one_gpu": summary(reps["one_gpu"], "whole frame on one GPU (every rank at once)"),
            "partitioned": summary(reps.get("partitioned"), "N-GPU partition: partitioned G-Buffer and Shadow Map Passes, SSAO and composition on bands")}

        # ---- the push kernel alone, from a profile of a few partitioned passes --------------------------------------------------------
        push_us = NOT_MEASURED
        if world > 1:
            mctx = map_context(scenes.sponza_like(min(tri_counts), seed=3))
            set_light(mctx, sc, np.zeros((4, 4), np.float32))
            for _ in range(3):
                map_pass(mctx, True)
            stream.synchronize()
            barrier()
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(20):
                    map_pass(mctx, True)
                stream.synchronize()
            ev = [e for e in prof.events() if "shadow_push_kernel" in e.name and e.device_type.name == "CUDA"]
            us = float(np.median([e.device_time for e in ev])) if ev else float("nan")
            push_us = {"us_max_over_ranks": reduce(us, dist.ReduceOp.MAX), "us_min_over_ranks": reduce(us, dist.ReduceOp.MIN), "kernels": len(ev)}
            barrier()
            mctx.close()
        rows_owned = sum(min(8, S - b * 8) for b in range((S + 7) // 8) if world > 1 and b % world == rank)
        result["push_kernel"] = {"time": push_us, "bytes_stored_per_rank": 4.0 * S * rows_owned * (world - 1) if world > 1 else 0.0}
    stream.synchronize()
    barrier()
    if rank == 0:
        print(json.dumps(result), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")
    fctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
