"""Multi-GPU execution of the hot path: one process per GPU (torch.distributed), scene + BVH replicated.

Two partitionings (SURVEY §8e):

* independent views (BASELINE config 5): view v -> rank v mod N, no data-path collective. That is what bench.py runs for
  N > 1 (weak scaling); nothing in this file is needed for it beyond `views_for_rank`.

* row bands of ONE frame (BASELINE config 4): rank r owns rows [y0, y1). The ray pass is per pixel and needs nothing
  from the neighbours. SVGF needs halo rows:
      temporal      reads history / moments / prev-normals at motion-displaced rows  -> `motion_halo` rows
      a-trous i     reads its input at rows +-2*2^i (and +-1 for the 3x3 variance gaussian) -> ATROUS_HALO[i] rows
  Every image lives full-size on every rank (memory is trivial next to 180 GB); a rank computes only its band and the
  rows it misses arrive by NCCL send/recv with the two neighbours, grouped per exchange (`HaloExchanger`). The G-buffer
  is an input of the path: each rank is given (or renders) band + GBUFFER_HALO rows of it.

The band driver (`RowBandSvgf`) is written against a small backend interface so that the SAME sequencing/halo logic runs
on the GPU (C-ABI backend below) and, in tests, on CPU tensors over gloo with the oracle as the per-band operator
(tests/test_multi_gpu_gloo.py): the halo widths and exchange order are what those tests pin.
"""
import numpy as np

ATROUS_ITERATIONS = 5
# rows of iteration i's INPUT needed beyond the band: taps at +-2*step rows (svgf_atrous_filter.comp:73), the variance
# gaussian at +-1 (svgf_atrous_filter.comp:24-27)
ATROUS_HALO = [max(2 * (1 << i), 1) for i in range(ATROUS_ITERATIONS)]      # 2, 4, 8, 16, 32
GBUFFER_HALO = 64       # normals are read at the a-trous taps of the widest iteration (32 rows) + the motion halo


def band_rows(height, world, rank):
    """Rows [y0, y1) of `rank`: contiguous, sizes differ by at most one row."""
    base, rem = divmod(height, world)
    y0 = rank * base + min(rank, rem)
    return y0, y0 + base + (1 if rank < rem else 0)


def required_motion_halo(motion_y_max_uv, height):
    """Rows of last frame's history / moments / normals the temporal pass can reach outside a band: svgf.comp:52 reprojects to
    coords - motion * size + 0.5 and the 3x3 retry (:81-97) looks one more texel around it. `motion_y_max_uv` is max |motion.y|
    over the frame (in UV units, as stored in the G-buffer)."""
    return int(np.ceil(float(motion_y_max_uv) * height)) + 2


def views_for_rank(n_views, world, rank):
    """Batch-of-views partition (config 5): round-robin."""
    return list(range(rank, n_views, world))


class HaloExchanger:
    """Exchanges `halo` boundary rows of a full-size row-major image with the ranks above and below.

    `image` is a torch tensor whose dim 0 is the image row (any device; NCCL for CUDA tensors, gloo for CPU ones).
    After `exchange`, rows [y0-halo, y0) hold the upper neighbour's last rows and [y1, y1+halo) the lower neighbour's
    first rows (clipped to the image and to what the neighbour actually owns)."""

    def __init__(self, height, world, rank, group=None):
        self.H, self.world, self.rank, self.group = height, world, rank, group
        self.y0, self.y1 = band_rows(height, world, rank)
        self.bytes_sent = 0
        self.exchanges = 0

    def _plan(self, halo):
        """[(peer, send_rows, recv_rows)] — a neighbour may own fewer than `halo` rows; then only its rows move and the
        rest of the halo comes from the rank beyond it (multi-hop halos are covered by looping over distance)."""
        plan = []
        for direction in (-1, +1):
            need = halo
            peer = self.rank + direction
            # rows I need beyond my band, walking outwards over as many neighbours as it takes
            edge = self.y0 if direction < 0 else self.y1
            while need > 0 and 0 <= peer < self.world:
                p0, p1 = band_rows(self.H, self.world, peer)
                take = min(need, p1 - p0)
                recv = (edge - take, edge) if direction < 0 else (edge, edge + take)
                plan.append((peer, None, recv))
                edge = recv[0] if direction < 0 else recv[1]
                need -= take
                peer += direction
        # what the others need from me: symmetric — rank q at distance d needs my rows closest to it
        for q in range(self.world):
            if q == self.rank:
                continue
            q0, q1 = band_rows(self.H, self.world, q)
            if q < self.rank:          # q is above me: it needs rows just below its band, i.e. [q1, q1+halo) ∩ mine
                lo, hi = max(self.y0, q1), min(self.y1, q1 + halo)
            else:                      # q is below me: it needs [q0-halo, q0) ∩ mine
                lo, hi = max(self.y0, q0 - halo), min(self.y1, q0)
            if hi > lo:
                plan.append((q, (lo, hi), None))
        return plan

    def exchange(self, images, halo):
        """`images`: list of tensors exchanged with the same halo in ONE grouped batch (one NCCL group launch)."""
        import torch.distributed as dist
        if self.world == 1 or halo <= 0:
            return
        ops, plan = [], self._plan(halo)
        # deterministic pairing order on both sides: sort by peer, sends before recvs for lower peer ids
        for img in images:
            for peer, send, recv in sorted(plan, key=lambda t: (t[0], t[1] is None)):
                if send is not None:
                    view = img[send[0]:send[1]]
                    ops.append(dist.P2POp(dist.isend, view, peer, group=self.group))
                    self.bytes_sent += view.numel() * view.element_size()
                else:
                    ops.append(dist.P2POp(dist.irecv, img[recv[0]:recv[1]], peer, group=self.group))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
            self.exchanges += 1


class RowBandSvgf:
    """SVGF Denoise Pass of hybrid_render_path.cpp:288-330 on a row band, halo exchanges interleaved.

    backend interface (all row ranges are [y0, y1) of the full image):
        temporal(rows)                 svgf.comp on `rows`; reads history/moments/prev-normals, writes integrated[0] + moments
        atrous(i, rows)                iteration i (step 2^i) on `rows`: integrated[0] -> integrated[1]
        copy_rows(src, dst, rows)      blit restricted to rows; names: "integ0", "integ1", "history", "normals", "prev_normals", "denoised"
        swap_integrated()              the ping-pong swap (:318, :328)
        tensor(name)                   torch tensor (rows first) aliasing the image, for the exchange
    """

    def __init__(self, backend, height, world, rank, motion_halo=8, group=None):
        self.b, self.H, self.world, self.rank = backend, height, world, rank
        self.y0, self.y1 = band_rows(height, world, rank)
        self.motion_halo = motion_halo
        self.x = HaloExchanger(height, world, rank, group)

    def _grown(self, halo):
        return max(0, self.y0 - halo), min(self.H, self.y1 + halo)

    def run(self):
        b, band = self.b, (self.y0, self.y1)
        # temporal accumulation on the band; its taps into last frame's history / moments / prev-normals reach at most
        # motion_halo rows outside, which the previous frame's exchanges below have already delivered
        b.temporal(band)
        # iteration 0 needs 2 rows of the temporal output beyond the band; next frame's temporal needs this frame's moments
        self.x.exchange([b.tensor("integ0")], ATROUS_HALO[0])
        self.x.exchange([b.tensor("moments")], self.motion_halo)
        for i in range(ATROUS_ITERATIONS):
            b.atrous(i, band)
            if i == 0:
                # iteration 0's output is both iteration 1's input (halo 4) and next frame's history (motion halo)
                h = max(ATROUS_HALO[1], self.motion_halo)
                self.x.exchange([b.tensor("integ1")], h)
                b.copy_rows("integ1", "history", self._grown(h))
            elif i < ATROUS_ITERATIONS - 1:
                self.x.exchange([b.tensor("integ1")], ATROUS_HALO[i + 1])
            # the last iteration's output is never read (SURVEY Q1): no exchange
            b.swap_integrated()
        b.copy_rows("normals", "prev_normals", self._grown(self.motion_halo))
        b.copy_rows("integ1", "denoised", band)       # after the swaps [1] is iteration 3's output
        b.swap_integrated()


# ---------------------------------------------------------------------------------------------------------------------
# Fused partition: no collective in the frame. Kernels store into the other ranks' images over NVLink (CUDA IPC peer
# memory) and the library orders the streams with flag words (include/vhr_b200.h, "one frame over several GPUs").
# torch.distributed only carries the IPC handles at set-up.
# ---------------------------------------------------------------------------------------------------------------------
def _has_image(ctx, name):
    from . import capi
    try:
        ctx.image_info(name)
        return True
    except capi.VhrError:
        return False


def _gbuffer_names(path):
    from . import hybrid_path as HP
    return [g[k] for g in path.gsets for k in (HP.N_ALBEDO, HP.N_NORMALS, HP.N_MOTION, HP.N_DEPTH)]


def _check_output_rank(ctxs, world, output_rank):
    """output_rank must name a rank, and RENDER_OUTPUT must exist on every context before it can be exported or attached"""
    from . import hybrid_path as HP
    if not 0 <= output_rank < world:
        raise ValueError(f"output_rank {output_rank} is not a rank of the partition (world {world})")
    for ctx in ctxs:
        if not _has_image(ctx, HP.N_RENDER_OUTPUT):
            raise ValueError(f"output_rank: {HP.N_RENDER_OUTPUT!r} is not actualized on this context; create it before the partition "
                             "(HybridRenderPath(..., composition=<format>), or ctx.actualize_image for the ray-traced path)")


def setup_fused_partition(ctx, path, world, rank, group=None, motion_halo=8, ray_block_rows=8, exchange_gbuffer=False,
                          exchange_shadow_map=False, output_rank=None):
    """Exports this rank's exchanged images, attaches everybody else's, installs the row partition on `ctx`.

    Exchanged images: the ray pass outputs (every rank stores into every owner's), the two integrated ping-pong images and
    the moments image with its twin (boundary rows pushed to the two neighbours). After this the plain single-GPU call
    sequence (`HybridRenderPath.frame`) runs the partitioned frame.
    exchange_gbuffer: also the four images of every G-buffer set, attached for all ranks, so that `HybridRenderPath.gbuffer_pass`
    runs partitioned (every rank traces its rows and stores them into every rank's G-buffer): the frame is driven from a camera.
    exchange_shadow_map: also the "Shadow Map", attached for all ranks, so that `HybridRenderPath.shadow_map_pass` runs partitioned
    (every rank rasterises its 8-row blocks of the map and stores them into every rank's map).
    output_rank: also rank `output_rank`'s RENDER_OUTPUT, attached on every other rank, and VHR_OPT_OUTPUT_RANK on every rank, so that
    the composition draws gather the whole frame into that rank's RENDER_OUTPUT. RENDER_OUTPUT must already exist on every rank."""
    import torch.distributed as dist
    from . import capi, hybrid_path as HP
    if output_rank is not None:
        _check_output_rank([ctx], world, output_rank)
    pc = path.pc
    mine = {"sync": ctx.sync_export_ipc(), "rt": [], "integ": [], "moments": None}
    for rt_name, refl_name in path.rt_sets:
        mine["rt"].append((ctx.image_export_ipc(rt_name), ctx.image_export_ipc(refl_name)))
    mine["gbuffer"] = [ctx.image_export_ipc(n) for n in _gbuffer_names(path)] if exchange_gbuffer else []
    mine["shadow_map"] = ctx.image_export_ipc(HP.N_SHADOW_MAP) if exchange_shadow_map else None
    mine["render_output"] = ctx.image_export_ipc(HP.N_RENDER_OUTPUT) if output_rank == rank else None
    for slot in pc["integrated_shadow_and_ao"]:
        mine["integ"].append((int(slot), ctx.storage_image_export_ipc(int(slot))[0]))
    mslot = int(pc["shadow_and_ao_moments_history"])
    mine["moments"] = (mslot,) + ctx.storage_image_export_ipc(mslot, twin=True)
    has_ssao = _has_image(ctx, "Screen Space Ambient Occlusion Raw")
    mine["ssao_raw"] = ctx.image_export_ipc("Screen Space Ambient Occlusion Raw") if has_ssao else None
    ctx.synchronize()
    everyone = [None] * world
    dist.all_gather_object(everyone, mine, group=group)
    for r, other in enumerate(everyone):
        if r == rank:
            continue
        ctx.sync_attach_peer(r, other["sync"])
        for (rt_name, refl_name), (h_rt, h_refl) in zip(path.rt_sets, other["rt"]):
            ctx.image_attach_peer(rt_name, r, h_rt)
            ctx.image_attach_peer(refl_name, r, h_refl)
        for name, h in zip(_gbuffer_names(path), other["gbuffer"]):
            ctx.image_attach_peer(name, r, h)
        if other["shadow_map"] is not None:
            ctx.image_attach_peer(HP.N_SHADOW_MAP, r, other["shadow_map"])
        if other["render_output"] is not None:
            ctx.image_attach_peer(HP.N_RENDER_OUTPUT, r, other["render_output"])
        if abs(r - rank) == 1:                       # halos only ever go to the two neighbours
            for (slot, _), (_, h) in zip(mine["integ"], other["integ"]):
                ctx.storage_image_attach_peer(slot, r, h)
            ctx.storage_image_attach_peer(mslot, r, other["moments"][1], other["moments"][2])
            if has_ssao and other["ssao_raw"]:
                ctx.image_attach_peer("Screen Space Ambient Occlusion Raw", r, other["ssao_raw"])
    bands = [band_rows(path.H, world, r)[0] for r in range(world)] + [path.H]
    ctx.set_partition(world, rank, bands, ray_block_rows=ray_block_rows, motion_halo=motion_halo)
    if output_rank is not None:
        ctx.set_option(capi.OPT_OUTPUT_RANK, output_rank)
    dist.barrier(group=group)                        # nobody starts storing into a peer that has not attached yet
    return bands


def setup_fused_partition_inprocess(ctxs, paths, motion_halo=8, ray_block_rows=8, exchange_gbuffer=False, exchange_shadow_map=False,
                                    output_rank=None):
    """The same partition for ranks that live in ONE process (one context per rank, all driven by this thread): peers are
    attached by plain device pointer. With all contexts on one GPU this exercises the whole fused path — interleaved ray
    blocks, halo pushes, flag-word ordering between the streams — on a single-GPU box (tests/test_partition_gpu.py).
    exchange_gbuffer, exchange_shadow_map, output_rank: as for setup_fused_partition."""
    from . import capi, hybrid_path as HP
    L = capi.lib()
    world = len(ctxs)
    H = paths[0].H
    if output_rank is not None:
        _check_output_rank(ctxs, world, output_rank)
    for r, (ctx, path) in enumerate(zip(ctxs, paths)):
        for q, (octx, opath) in enumerate(zip(ctxs, paths)):
            if q == r:
                continue
            capi._check(L.vhr_sync_attach_peer_pointer(ctx._h, q, L.vhr_sync_device_ptr(octx._h)))
            for (rt_name, refl_name), (ort, orefl) in zip(path.rt_sets, opath.rt_sets):
                capi._check(L.vhr_image_attach_peer_pointer(ctx._h, rt_name.encode(), q, octx.image_info(ort)[0]))
                capi._check(L.vhr_image_attach_peer_pointer(ctx._h, refl_name.encode(), q, octx.image_info(orefl)[0]))
            if exchange_gbuffer:
                for name, oname in zip(_gbuffer_names(path), _gbuffer_names(opath)):
                    capi._check(L.vhr_image_attach_peer_pointer(ctx._h, name.encode(), q, octx.image_info(oname)[0]))
            if exchange_shadow_map:
                capi._check(L.vhr_image_attach_peer_pointer(ctx._h, HP.N_SHADOW_MAP.encode(), q, octx.image_info(HP.N_SHADOW_MAP)[0]))
            if q == output_rank:
                capi._check(L.vhr_image_attach_peer_pointer(ctx._h, HP.N_RENDER_OUTPUT.encode(), q, octx.image_info(HP.N_RENDER_OUTPUT)[0]))
            if abs(q - r) == 1:
                for slot, oslot in zip(path.pc["integrated_shadow_and_ao"], opath.pc["integrated_shadow_and_ao"]):
                    capi._check(L.vhr_storage_image_attach_peer_pointer(ctx._h, int(slot), q, octx.storage_image_info(int(oslot))[0], None))
                ms, oms = int(path.pc["shadow_and_ao_moments_history"]), int(opath.pc["shadow_and_ao_moments_history"])
                L.vhr_storage_image_twin_device_ptr(ctx._h, ms)          # allocate my own twin before anybody swaps
                capi._check(L.vhr_storage_image_attach_peer_pointer(ctx._h, ms, q, octx.storage_image_info(oms)[0],
                                                                    L.vhr_storage_image_twin_device_ptr(octx._h, oms)))
                if _has_image(ctx, "Screen Space Ambient Occlusion Raw") and _has_image(octx, "Screen Space Ambient Occlusion Raw"):
                    capi._check(L.vhr_image_attach_peer_pointer(ctx._h, b"Screen Space Ambient Occlusion Raw", q,
                                                                octx.image_info("Screen Space Ambient Occlusion Raw")[0]))
    bands = [band_rows(H, world, r)[0] for r in range(world)] + [H]
    for r, ctx in enumerate(ctxs):
        ctx.set_partition(world, r, bands, ray_block_rows=ray_block_rows, motion_halo=motion_halo)
        if output_rank is not None:
            ctx.set_option(capi.OPT_OUTPUT_RANK, output_rank)
    return bands


# ---------------------------------------------------------------------------------------------------------------------
# GPU backend over the C-ABI
# ---------------------------------------------------------------------------------------------------------------------
class _DeviceRows:
    """__cuda_array_interface__ view of a dense fp16 image: shape (rows, row_elems)."""

    def __init__(self, ptr, rows, row_elems):
        self.__cuda_array_interface__ = {"shape": (rows, row_elems), "typestr": "<f2", "data": (int(ptr), False), "version": 3}


class CabiBandBackend:
    """Drives libvhr_b200.so for one rank's band (images full-size, dispatches restricted with VHR_OPT_ROW_BEGIN/END)."""

    def __init__(self, ctx, path, gset=0):
        from . import capi, hybrid_path as HP
        self.capi, self.HP, self.ctx, self.path, self.gset = capi, HP, ctx, path, gset
        self.W, self.H = path.W, path.H
        self._tensors = {}

    def _rows(self, rows):
        self.ctx.set_option(self.capi.OPT_ROW_BEGIN, rows[0])
        self.ctx.set_option(self.capi.OPT_ROW_END, rows[1])

    def _bind(self):
        HP, g = self.HP, self.path.gsets[self.gset]
        self.ctx.bind_pass_images([g[HP.N_NORMALS], g[HP.N_MOTION], g[HP.N_DEPTH], HP.N_RT, HP.N_DENOISED])

    def trace(self, rows):
        self._rows(rows)
        self.path.raytrace_pass(self.gset)

    def temporal(self, rows):
        self._rows(rows)
        self._bind()
        self.ctx.dispatch(self.HP.SHADER_SVGF, self.HP.groups(self.W), self.HP.groups(self.H), 1, self.path.pc)

    def atrous(self, i, rows):
        self._rows(rows)
        self.path.pc["atrous_step"] = 1 << i
        self.ctx.dispatch(self.HP.SHADER_ATROUS, self.HP.groups(self.W), self.HP.groups(self.H), 1, self.path.pc)

    def swap_integrated(self):
        pc = self.path.pc
        pc["integrated_shadow_and_ao"] = pc["integrated_shadow_and_ao"][::-1].copy()

    def _resolve(self, name):
        """name -> (device pointer, elements per row)"""
        HP, pc, g = self.HP, self.path.pc, self.path.gsets[self.gset]
        if name in ("integ0", "integ1"):
            p, w, h, f = self.ctx.storage_image_info(int(pc["integrated_shadow_and_ao"][int(name[-1])]))
        elif name == "history":
            p, w, h, f = self.ctx.storage_image_info(int(pc["shadow_and_ao_history"]))
        elif name == "moments":
            p, w, h, f = self.ctx.storage_image_info(int(pc["shadow_and_ao_moments_history"]))
        elif name == "prev_normals":
            p, w, h, f = self.ctx.storage_image_info(int(pc["prev_frame_normals_and_object_ids"]))
        elif name == "normals":
            p, w, h, f = self.ctx.image_info(g[HP.N_NORMALS])
        elif name == "denoised":
            p, w, h, f = self.ctx.image_info(HP.N_DENOISED)
        elif name == "rt":
            p, w, h, f = self.ctx.image_info(HP.N_RT)
        else:
            raise KeyError(name)
        return p, w * HP.T.FORMAT_TEXEL_BYTES[f] // 2

    def tensor(self, name):
        import torch
        p, row_elems = self._resolve(name)
        key = (int(p), row_elems)
        if key not in self._tensors:
            self._tensors[key] = torch.as_tensor(_DeviceRows(p, self.H, row_elems), device="cuda")
        return self._tensors[key]

    def copy_rows(self, src, dst, rows):
        s, d = self.tensor(src), self.tensor(dst)
        d[rows[0]:rows[1]].copy_(s[rows[0]:rows[1]], non_blocking=True)
