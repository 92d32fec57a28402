"""Multi-GPU host logic (one process per GPU, torch.distributed for the plumbing).

Batch sharding (BASELINE config C3; SURVEY.md §8e): images are independent through the decoder
(GroupNorm is per sample), but every global statistic of the HDR epilogue is taken over the WHOLE
batch (hdr_vae_decode.py:862-865,1098,1116; SURVEY.md §0.7).  So the path has exactly one exchange
step: between epilogue phase A and phase B the raw statistics block (4 mins, 4 maxes, 8 sums) is
all-reduced, after which every rank finishes its own images with identical scalars — results do
not depend on the number of GPUs."""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch
import torch.distributed as dist


def shard_bounds(n_items: int, world_size: int) -> List[Tuple[int, int]]:
    """Contiguous, balanced [start, end) ranges; the first n_items % world ranks get one extra."""
    if world_size < 1:
        raise ValueError("world_size must be >= 1")
    base, extra = divmod(n_items, world_size)
    out, s = [], 0
    for r in range(world_size):
        e = s + base + (1 if r < extra else 0)
        out.append((s, e))
        s = e
    return out


def allreduce_raw_stats(vmin: torch.Tensor, vmax: torch.Tensor, vsum: torch.Tensor, group=None) -> None:
    """In-place cross-rank reduction of an hdrvae_raw_stats block (include/hdrvae.h): MIN / MAX / SUM, as three
    all-reduces.  Used for host-side (CPU / gloo) blocks and by the row-tiling executor; the batch-sharded GPU path
    uses :func:`exchange_raw_stats_block` (ONE all-gather + a fixed-order merge kernel)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    dist.all_reduce(vmin, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(vmax, op=dist.ReduceOp.MAX, group=group)
    dist.all_reduce(vsum, op=dist.ReduceOp.SUM, group=group)


def merge_raw_stats(blocks: Sequence[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]):
    """Single-process equivalent of :func:`allreduce_raw_stats` (tests / emulation)."""
    vmin = torch.stack([b[0] for b in blocks]).amin(0)
    vmax = torch.stack([b[1] for b in blocks]).amax(0)
    vsum = torch.stack([b[2] for b in blocks]).sum(0)
    return vmin, vmax, vsum


RAW_BLOCK_BYTES = 96
_gather_bufs = {}


def identity_raw_block(device) -> torch.Tensor:
    """The neutral hdrvae_raw_stats block (+inf mins, -inf maxes, zero sums) a rank with an EMPTY shard contributes."""
    blk = torch.zeros(RAW_BLOCK_BYTES, dtype=torch.uint8, device=device)
    blk[0:16].view(torch.float32).fill_(float("inf"))
    blk[16:32].view(torch.float32).fill_(float("-inf"))
    return blk


def exchange_raw_stats_block(block: torch.Tensor, lib=None, group=None) -> None:
    """The ONE exchange step of batch sharding: all-gather every rank's 96-byte block (one NCCL collective), then merge
    the gathered blocks in rank order into `block` (uint8[96] view of the workspace) with one kernel
    (hdrvae_raw_stats_merge) — every rank ends with bit-identical statistics.  CPU tensors (gloo tests) are merged
    with torch ops in the same order."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    world = dist.get_world_size(group)
    key = (block.device, world)
    buf = _gather_bufs.get(key)
    if buf is None:
        buf = _gather_bufs[key] = torch.empty(world * RAW_BLOCK_BYTES, dtype=torch.uint8, device=block.device)
    dist.all_gather_into_tensor(buf, block, group=group)
    if block.is_cuda:
        from . import _native as N
        lib = lib or N.load_library()
        N.check(lib.hdrvae_raw_stats_merge(buf.data_ptr(), world, block.data_ptr(),
                                           torch.cuda.current_stream(block.device).cuda_stream), "hdrvae_raw_stats_merge")
    else:
        rows = buf.view(world, RAW_BLOCK_BYTES)
        vmin = rows[:, 0:16].contiguous().view(torch.float32).view(world, 4).amin(0)
        vmax = rows[:, 16:32].contiguous().view(torch.float32).view(world, 4).amax(0)
        vs = rows[:, 32:96].contiguous().view(torch.float64).view(world, 8)
        vsum = vs[0].clone()
        for r in range(1, world):
            vsum += vs[r]
        block[0:16].view(torch.float32).copy_(vmin)
        block[16:32].view(torch.float32).copy_(vmax)
        block[32:96].view(torch.float64).copy_(vsum)


_validated = set()


def _validate_across_ranks(latent_local: torch.Tensor, hdr_mode: str, ev_multiplier: float, group) -> None:
    """Once per (shape, mode, multiplier, group): every rank must decode the same latent shape (apart from the batch
    count) with the same mode and multiplier, otherwise the batch-global statistics would be meaningless."""
    sig = (tuple(latent_local.shape[1:]), str(hdr_mode).lower(), float(ev_multiplier))
    key = (sig, id(group))
    if key in _validated:
        return
    sigs = [None] * dist.get_world_size(group)
    dist.all_gather_object(sigs, sig, group=group)
    if any(s != sigs[0] for s in sigs):
        raise ValueError(f"decode_batch_sharded: ranks disagree on latent shape / mode / multiplier: {sigs}")
    _validated.add(key)


def decode_batch_sharded(engine, latent_local: torch.Tensor, hdr_mode: str, ev_multiplier: float = 1.0, group=None,
                         want_stats: bool = True):
    """Decode this rank's slice of the batch with batch-global HDR statistics.

    engine: vae_decode_hdr_b200.engine.HdrVaeEngine on this rank's GPU.  Returns (image_local, stats)
    where the pre/post/conv/pre3 statistics and every derived scalar are those of the whole batch;
    out_min/out_max/hdr_pixels describe the local slice.  A rank whose slice is EMPTY (batch smaller than the world
    size, shard_bounds) skips the decoder, contributes the neutral block to the exchange and returns an empty image."""
    distributed = dist.is_initialized() and dist.get_world_size(group) > 1
    if distributed:
        _validate_across_ranks(latent_local, hdr_mode, ev_multiplier, group)
    # after the validation: every rank holds the same shape, so either all ranks raise here or none does
    if latent_local.dim() != 4 or latent_local.shape[1] != engine.latent_channels:
        raise ValueError(f"expected a latent [B,{engine.latent_channels},h,w] for this VAE, got {tuple(latent_local.shape)}")
    if latent_local.shape[0] == 0:
        if distributed:
            exchange_raw_stats_block(identity_raw_block(engine.device), engine.lib, group)
        h, w = latent_local.shape[2:]
        return torch.empty((0, 8 * h, 8 * w, 3), dtype=torch.float32, device=engine.device), None
    # The library replays the two halves of the decode as CUDA graphs, which needs a non-default stream: hop to the
    # engine's stream when the caller sits on the legacy default stream (the NCCL collective follows torch's current
    # stream, so it is ordered between the two graphs either way).
    cur = torch.cuda.current_stream(engine.device)
    if cur.cuda_stream != 0:
        block = engine.decode_begin_block(latent_local)
        exchange_raw_stats_block(block, engine.lib, group)
        return engine.decode_finish(hdr_mode, ev_multiplier, want_stats)
    side = engine._side
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        latent_local.record_stream(side)
        block = engine.decode_begin_block(latent_local)
        exchange_raw_stats_block(block, engine.lib, group)
        out, st = engine.decode_finish(hdr_mode, ev_multiplier, want_stats)
    cur.wait_stream(side)
    out.record_stream(cur)
    return out, st


# ------------------------------------------------------------------------------------------------ row tiling
# One image, latent rows split evenly over the ranks (BASELINE config C4).  libhdrvae runs the same step program
# on every rank's slab and tells the host what to exchange between steps (include/hdrvae.h, hdrvae_exchange):
# 1-row conv halos to the neighbours, GroupNorm sums all-reduced, attention K/V all-gathered, HDR statistics
# all-reduced.  Here the exchanges are NCCL collectives / point-to-point (torch.distributed) on views of the
# workspace; `decode_rows_emulated` performs the same exchanges with plain copies between R workspaces of ONE
# process, which is how the path is tested on a single GPU.
import ctypes as C  # noqa: E402

from . import _native as _N  # noqa: E402


def _raw_views(ws: torch.Tensor, off: int):
    blk = ws[off:off + 96]
    return blk[0:16].view(torch.float32), blk[16:32].view(torch.float32), blk[32:96].view(torch.float64)


def _exchange_nccl(ex, ws: torch.Tensor, rank: int, world: int, group=None) -> None:
    if ex.kind & _N.EX_HALO:
        ops = []
        for i in range(ex.n_halo):
            n = ex.halo_row_bytes[i]
            first, last = ws[ex.halo_first_row_off[i]:ex.halo_first_row_off[i] + n], ws[ex.halo_last_row_off[i]:ex.halo_last_row_off[i] + n]
            top, bot = ws[ex.halo_top_off[i]:ex.halo_top_off[i] + n], ws[ex.halo_bottom_off[i]:ex.halo_bottom_off[i] + n]
            if rank > 0:
                ops += [dist.P2POp(dist.isend, first, rank - 1, group), dist.P2POp(dist.irecv, top, rank - 1, group)]
            if rank < world - 1:
                ops += [dist.P2POp(dist.isend, last, rank + 1, group), dist.P2POp(dist.irecv, bot, rank + 1, group)]
        if ops:
            for r in dist.batch_isend_irecv(ops):
                r.wait()
    if ex.kind & _N.EX_ALLREDUCE_F64:
        buf = ws[ex.allreduce_off:ex.allreduce_off + 8 * ex.allreduce_count].view(torch.float64)
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    if ex.kind & _N.EX_ALLGATHER:
        for i in range(ex.n_gather):
            n = ex.gather_bytes_per_rank[i]
            full = ws[ex.gather_off[i]:ex.gather_off[i] + n * world]
            dist.all_gather_into_tensor(full, full[rank * n:(rank + 1) * n].clone(), group=group)
    if ex.kind & _N.EX_RAW_STATS:
        allreduce_raw_stats(*_raw_views(ws, ex.raw_stats_off), group=group)


def decode_rows_sharded(engine, latent_full: torch.Tensor, hdr_mode: str, ev_multiplier: float = 1.0, group=None,
                        want_stats: bool = True):
    """Row-tiled decode of ONE image across the ranks of `group`: returns this rank's rows of the image
    ([1, 8h/world, 8w, 3]) and the statistics (pre/post/conv/pre3 global, out_* of the local slab)."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    state, ws, out, _keep = engine.rows_begin(latent_full, rank, world, hdr_mode, ev_multiplier)
    while True:
        ex = engine.rows_run(state)
        if ex.kind == _N.EX_END:
            break
        _exchange_nccl(ex, ws, rank, world, group)
    return out, engine.rows_end(state, want_stats)


def decode_rows_emulated(engine, latent_full: torch.Tensor, world: int, hdr_mode: str, ev_multiplier: float = 1.0):
    """The same row-tiled program with `world` virtual ranks on ONE GPU (one workspace each, run in lock step);
    exchanges are device copies.  Returns the full image [1, 8h, 8w, 3] and rank 0's statistics."""
    states, wss, outs, keep = [], [], [], []
    for r in range(world):
        st, ws, out, z = engine.rows_begin(latent_full, r, world, hdr_mode, ev_multiplier)
        states.append(st); wss.append(ws); outs.append(out); keep.append(z)
    while True:
        exs = [engine.rows_run(st) for st in states]
        ex = exs[0]
        if ex.kind == _N.EX_END:
            break
        if ex.kind & _N.EX_HALO:
            for i in range(ex.n_halo):
                n = ex.halo_row_bytes[i]
                for r in range(world):
                    if r > 0:       # my first interior row -> upper neighbour's bottom halo
                        wss[r - 1][ex.halo_bottom_off[i]:ex.halo_bottom_off[i] + n].copy_(wss[r][ex.halo_first_row_off[i]:ex.halo_first_row_off[i] + n])
                    if r < world - 1:   # my last interior row -> lower neighbour's top halo
                        wss[r + 1][ex.halo_top_off[i]:ex.halo_top_off[i] + n].copy_(wss[r][ex.halo_last_row_off[i]:ex.halo_last_row_off[i] + n])
        if ex.kind & _N.EX_ALLREDUCE_F64:
            views = [ws[ex.allreduce_off:ex.allreduce_off + 8 * ex.allreduce_count].view(torch.float64) for ws in wss]
            total = torch.stack(views).sum(0)
            for v in views:
                v.copy_(total)
        if ex.kind & _N.EX_ALLGATHER:
            for i in range(ex.n_gather):
                n = ex.gather_bytes_per_rank[i]
                parts = [wss[r][ex.gather_off[i] + r * n:ex.gather_off[i] + (r + 1) * n].clone() for r in range(world)]
                for ws in wss:
                    for r in range(world):
                        ws[ex.gather_off[i] + r * n:ex.gather_off[i] + (r + 1) * n].copy_(parts[r])
        if ex.kind & _N.EX_RAW_STATS:
            blocks = [_raw_views(ws, ex.raw_stats_off) for ws in wss]
            vmin, vmax, vsum = merge_raw_stats(blocks)
            for b in blocks:
                b[0].copy_(vmin); b[1].copy_(vmax); b[2].copy_(vsum)
    stats = [engine.rows_end(st, True) for st in states]
    return torch.cat(outs, dim=1), stats[0]


class RowsDirect:
    """Row-tiled decode with DEVICE-DRIVEN exchanges (csrc/rows_p2p.cu): every rank's workspace is allocated by the
    library and shared over CUDA IPC (hdrvae_peer_alloc / hdrvae_peer_open — no private torch API; torch.distributed is
    used once, to all-gather the 64-byte handles); `decode` then enqueues the WHOLE step program in one C call: at every
    exchange point a push kernel stores this rank's halo rows, GroupNorm sums, attention K / V rows and HDR statistics
    straight into the peers' workspaces over NVLink behind a two-phase flag handshake, and a wait kernel folds the sums in
    rank order.  No NCCL call and no host round trip on the data path (the NCCL transport returns to Python ~35 times per
    decode).  One process per GPU; the workspace is persistent, `decode` may be called any number of times for latents of
    the shape given at construction."""

    def __init__(self, engine, h: int, w: int, group=None):
        self.engine, self.group, self.h, self.w = engine, group, h, w
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        lib, ctx = engine.lib, engine._ctx
        self.bytes = engine.rows_workspace_bytes(h, w, self.world)
        self._own = C.c_void_p()
        handle = _N.HdrvaeIpcHandle()
        with torch.cuda.device(engine.device):
            _N.check(lib.hdrvae_peer_alloc(ctx, self.bytes, C.byref(self._own), C.byref(handle)), "hdrvae_peer_alloc")
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle.bytes), group=group)
        self._mapped = {}
        ptrs = (C.c_void_p * self.world)()
        for r in range(self.world):
            if r == self.rank:
                ptrs[r] = self._own.value
                continue
            h_r = _N.HdrvaeIpcHandle()
            C.memmove(h_r.bytes, handles[r], 64)
            m = C.c_void_p()
            _N.check(lib.hdrvae_peer_open(ctx, C.byref(h_r), C.byref(m)), "hdrvae_peer_open")
            self._mapped[r] = m
            ptrs[r] = m.value
        self._ptrs = ptrs
        dist.barrier(group=group)       # nobody starts pushing before every mapping exists

    def decode(self, latent_full: torch.Tensor, hdr_mode: str, ev_multiplier: float = 1.0, want_stats: bool = True):
        if tuple(latent_full.shape[-2:]) != (self.h, self.w):
            raise ValueError(f"this RowsDirect was built for {self.h}x{self.w} latents, got {tuple(latent_full.shape)}")
        eng = self.engine
        state, _ws, out, _keep = eng.rows_begin(latent_full, self.rank, self.world, hdr_mode, ev_multiplier,
                                                workspace=(self._own.value, self.bytes))
        _N.check(eng.lib.hdrvae_rows_set_peers(state, self._ptrs, self.world), "hdrvae_rows_set_peers")
        with torch.cuda.device(eng.device):
            _N.check(eng.lib.hdrvae_rows_run_direct(state, eng._stream()), "hdrvae_rows_run_direct")
        return out, eng.rows_end(state, want_stats)

    def close(self) -> None:
        """Collective: every rank must call it (a rank may only free its workspace once nobody maps it any more)."""
        if getattr(self, "_own", None) is None:
            return
        lib, ctx = self.engine.lib, self.engine._ctx
        torch.cuda.synchronize(self.engine.device)
        dist.barrier(group=self.group)
        for m in self._mapped.values():
            lib.hdrvae_peer_close(ctx, m)
        self._mapped = {}
        dist.barrier(group=self.group)
        lib.hdrvae_peer_free(ctx, self._own)
        self._own = None
