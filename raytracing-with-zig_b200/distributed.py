"""Multi-GPU: one process per GPU, image-space interleaved tiles, gather to rank 0.

north_star / SURVEY.md §8e: tile k of the frame belongs to rank k % world; every rank renders its
tiles into a compact buffer (equal size on every rank) and rank 0 collects them with ONE gather
over NCCL (NVLink/NVSwitch) and de-interleaves on the device.  The path has no other exchange:
every (pixel, sample) is independent once the RNG is counter based.
"""
from __future__ import annotations

import numpy as np

from . import binding as B

DEFAULT_TILE = (4, 4)  # measured on C3, max/mean shard time at 8 / 4 / 2 ranks: 1.004 / 1.001 / 1.000 (32x8: 1.023 / 1.011 / 1.009; tools/shard_balance.py)


def tile_index_map(width: int, height: int, world: int, tile_w: int, tile_h: int):
    """Host-side description of the tile layout (pure index arithmetic, used by tests and docs).

    Returns (per_rank_pixels, idx) where idx[y, x] is the position of pixel (x, y) in the
    concatenation of the `world` compact rank buffers.  Mirrors csrc deinterleave_kernel."""
    tiles_x = (width + tile_w - 1) // tile_w
    tiles_y = (height + tile_h - 1) // tile_h
    n_local_tiles = (tiles_x * tiles_y + world - 1) // world
    per_rank = n_local_tiles * tile_w * tile_h
    y, x = np.mgrid[0:height, 0:width]
    tx, ty = x // tile_w, y // tile_h
    gt = ty * tiles_x + tx
    rank, lt = gt % world, gt // world
    lp = lt * (tile_w * tile_h) + (y - ty * tile_h) * tile_w + (x - tx * tile_w)
    return per_rank, (rank * per_rank + lp).astype(np.int64)


def gather_tiles(local, world: int, rank: int, group=None):
    """Gather equal-sized compact tile buffers to rank 0 (torch.distributed: NCCL on GPUs, gloo on CPU).

    Returns the concatenated [world * n, 3] tensor on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist

    if world == 1:
        return local
    if rank == 0:
        gathered = torch.empty((world,) + tuple(local.shape), dtype=local.dtype, device=local.device)
        dist.gather(local, gather_list=list(gathered.unbind(0)), dst=0, group=group)
        return gathered.reshape(world * local.shape[0], *local.shape[1:])
    dist.gather(local, gather_list=None, dst=0, group=group)
    return None


def render_sharded(renderer, camera, tile=DEFAULT_TILE, group=None):
    """Camera.render across the ranks of the default process group.

    Every rank calls this with the same camera and an uploaded copy of the scene.  Returns
    (image [H,W,3] uint8 device tensor on rank 0 / None elsewhere, this rank's stats)."""
    import torch.distributed as dist

    rank, world = (dist.get_rank(group), dist.get_world_size(group)) if dist.is_initialized() else (0, 1)
    shard = B.rtz_shard(rank, world, tile[0], tile[1])
    local, st = renderer.render(camera, shard)
    gathered = gather_tiles(local, world, rank, group)
    if rank != 0:
        return None, st
    img = renderer.deinterleave(gathered, int(camera.width), int(camera.height), world, tile[0], tile[1])
    return img, st


def render_sharded_denoised(renderer, camera, guide_samples: int = 0, params=None, tile=DEFAULT_TILE, group=None):
    """`rtz_render_denoised` across the ranks of the default process group: every rank renders the linear colour
    and the guides of its tiles, rank 0 gathers the three float32 buffers, de-interleaves them and denoises the whole
    frame.  The camera must carry its seed (every rank has to trace the same rays).  Returns (uint8 [H,W,3],
    float32 [H,W,3] denoised device tensors on rank 0 / (None, None) elsewhere, this rank's render stats)."""
    import torch.distributed as dist

    if not camera.has_seed:
        raise ValueError("render_sharded_denoised needs a camera with its seed: every rank must trace the same rays")
    rank, world = (dist.get_rank(group), dist.get_world_size(group)) if dist.is_initialized() else (0, 1)
    spp = int(camera.samples_per_pixel)
    g = int(guide_samples) if guide_samples else min(spp, 16)
    shard = B.rtz_shard(rank, world, tile[0], tile[1])
    _, linear, st = renderer.render_linear(camera, shard)
    albedo, normal, _ = renderer.render_guides(camera, g, shard=shard)
    W, H = int(camera.width), int(camera.height)
    planes = []
    for local in (linear, albedo, normal):
        gathered = gather_tiles(local, world, rank, group)
        if rank == 0:
            planes.append(renderer.deinterleave(gathered, W, H, world, tile[0], tile[1]))
    if rank != 0:
        return None, None, st
    rgb, lin, _ = renderer.denoise(*planes, params=params)
    return rgb, lin, st
