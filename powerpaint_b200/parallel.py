"""Batch sharding across the GPUs of one box (SURVEY.md §8e): requests are independent, so a batch is
split contiguously (both CFG halves of an image stay on one rank), weights are replicated, and the only
communication is a scatter of the inputs before the loop and a gather of the decoded images after it —
no collective inside the denoising loop. One process per GPU; `torch.distributed` (NCCL over
NVLink/NVSwitch on GPUs, gloo in the CPU tests) is the plumbing.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch


def shard_ranges(total: int, world: int) -> List[Tuple[int, int]]:
    """contiguous [start, end) per rank; the first `total % world` ranks take one extra request"""
    if world <= 0:
        raise ValueError("world must be positive")
    base, rem = divmod(total, world)
    out, s = [], 0
    for r in range(world):
        n = base + (1 if r < rem else 0)
        out.append((s, s + n))
        s += n
    return out


def scatter_requests(tensors: Optional[Sequence[torch.Tensor]], shapes: Sequence[Tuple[int, ...]],
                     dtypes: Sequence[torch.dtype], device, src: int = 0, group=None) -> List[torch.Tensor]:
    """Rank `src` holds full-batch tensors [world * b, ...]; every rank receives its [b, ...] shard.
    `shapes`/`dtypes` describe ONE shard (known on all ranks)."""
    import torch.distributed as dist

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    out = []
    for k, (shape, dt) in enumerate(zip(shapes, dtypes)):
        dst = torch.empty(shape, dtype=dt, device=device)
        if rank == src:
            full = tensors[k].to(device)
            if full.shape[0] != world * shape[0]:
                raise ValueError(f"tensor {k}: batch {full.shape[0]} != world*shard {world * shape[0]}")
            chunks = [c.contiguous() for c in full.chunk(world, dim=0)]
        else:
            chunks = None
        dist.scatter(dst, chunks, src=src, group=group)
        out.append(dst)
    return out


def gather_images(images: torch.Tensor, dst: int = 0, group=None) -> Optional[torch.Tensor]:
    """every rank contributes [b, ...]; rank `dst` gets [world * b, ...] in rank order, others None"""
    import torch.distributed as dist

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    bufs = [torch.empty_like(images) for _ in range(world)] if rank == dst else None
    dist.gather(images.contiguous(), bufs, dst=dst, group=group)
    return torch.cat(bufs, dim=0) if rank == dst else None


def scatter_batch(tensors: Optional[Sequence[torch.Tensor]], device, src: int = 0, group=None) -> List[torch.Tensor]:
    """Ragged form of `scatter_requests`: rank `src` holds full-batch tensors [total, ...] (all with the same `total`;
    the other ranks pass None and need to know nothing), rank r receives rows `shard_ranges(total, world)[r]` of each —
    shards differ by at most one row and may be EMPTY when total < world (the caller skips its `__call__` then).
    One object broadcast carries the shapes / dtypes; the payload travels as equal-sized (padded) scatter chunks."""
    import torch.distributed as dist

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if rank == src:
        if not tensors:
            raise ValueError("rank `src` must pass the full-batch tensors")
        totals = {int(t.shape[0]) for t in tensors}
        if len(totals) != 1:
            raise ValueError(f"all tensors must share the batch dimension, got {sorted(totals)}")
        meta = [[(tuple(t.shape), t.dtype) for t in tensors]]
    else:
        meta = [None]
    dist.broadcast_object_list(meta, src=src, group=group)
    out = []
    for k, (shape, dt) in enumerate(meta[0]):
        total = shape[0]
        ranges = shard_ranges(total, world)
        rows = max(e - s for s, e in ranges)  # == ceil(total / world)
        s, e = ranges[rank]
        dst = torch.empty((rows,) + tuple(shape[1:]), dtype=dt, device=device)
        chunks = None
        if rank == src:
            full = tensors[k].to(device)
            chunks = []
            for cs, ce in ranges:
                c = torch.zeros_like(dst)
                c[: ce - cs] = full[cs:ce]
                chunks.append(c)
        if rows > 0:
            dist.scatter(dst, chunks, src=src, group=group)
        out.append(dst[: e - s].contiguous())
    return out


def gather_batch(local: torch.Tensor, total: int, dst: int = 0, group=None) -> Optional[torch.Tensor]:
    """inverse of `scatter_batch`: rank r contributes its `shard_ranges(total, world)[r]` rows (possibly none; shape
    [0, ...] with the right trailing dimensions and dtype), rank `dst` gets [total, ...] in rank order, others None"""
    import torch.distributed as dist

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    ranges = shard_ranges(total, world)
    s, e = ranges[rank]
    if local.shape[0] != e - s:
        raise ValueError(f"rank {rank} holds {local.shape[0]} rows, its shard of {total} over {world} ranks is {e - s}")
    rows = max(ce - cs for cs, ce in ranges)
    if rows == 0:
        return local if rank == dst else None
    send = torch.zeros((rows,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    send[: e - s] = local
    bufs = [torch.empty_like(send) for _ in range(world)] if rank == dst else None
    dist.gather(send, bufs, dst=dst, group=group)
    if rank != dst:
        return None
    return torch.cat([b[: ce - cs] for b, (cs, ce) in zip(bufs, ranges)], dim=0)


def _split_batched(batched: dict, total: int):
    """full-batch keywords -> (names, halves, tensors) to scatter; a [2 x total] keyword ([negative; positive], the
    BrushNet pipeline's `prompt_embedsU`) travels as two [total] tensors (halves 1 and 2) so that each half is sharded
    like the images; a list of [total] tensors (one control image per ControlNet) travels element by element
    (halves == 3); halves == 0 marks an ordinary [total] keyword"""
    names, halves, tensors = [], [], []
    for k, v in batched.items():
        if isinstance(v, (list, tuple)):
            for t in v:
                if t.shape[0] != total:
                    raise ValueError(f"`{k}`: batch {t.shape[0]} of a list entry is not the request's {total}")
                names.append(k), halves.append(3), tensors.append(t)
        elif v.shape[0] == total:
            names.append(k), halves.append(0), tensors.append(v)
        elif v.shape[0] == 2 * total:
            names += [k, k]
            halves += [1, 2]
            tensors += [v[:total], v[total:]]
        else:
            raise ValueError(f"`{k}`: batch {v.shape[0]} is neither the request's {total} nor twice it")
    return names, halves, tensors


def _merge_shards(names, halves, shards) -> dict:
    """inverse of `_split_batched` on one rank's shards: the two halves of a stacked keyword are concatenated again"""
    kw = {}
    for k, half, t in zip(names, halves, shards):
        if half == 3:
            kw.setdefault(k, []).append(t)
        else:
            kw[k] = torch.cat([kw[k], t]) if half == 2 else t
    return kw


def sharded_call(pipe, batched: Optional[dict], device, seeds: Optional[Sequence[int]] = None, src: int = 0,
                 group=None, **common) -> Optional[torch.Tensor]:
    """One request batch over all ranks: rank `src` passes `batched` = {`__call__` keyword: full-batch tensor [total, ...]}
    (image, mask, prompt_embeds, negative_prompt_embeds, control_image, ...; the other ranks pass None), every rank
    passes the same `common` keywords (height, width, num_inference_steps, guidance_scale, output_type = "uint8" |
    "latent" | "pt", ...). Each rank runs `pipe(...)` on its contiguous shard — no collective inside the call — and rank
    `src` gets the images of the whole batch in request order (others None). `seeds[i]` seeds the generator of GLOBAL
    image i, so the result does not depend on the number of ranks. A rank whose shard is empty skips the call.
    Keywords whose batch is 2 x total (the BrushNet pipeline's `prompt_embedsU` = [negative; positive]) are split per
    half; a list of full-batch tensors (`control_image` of several ControlNets) is scattered entry by entry and arrives
    as a list."""
    import torch.distributed as dist

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if rank == src:
        if not batched:
            raise ValueError("rank `src` must pass the batched keywords")
        first = batched["image"] if "image" in batched else next(iter(batched.values()))
        total = int((first[0] if isinstance(first, (list, tuple)) else first).shape[0])
        names, halves, tensors = _split_batched(batched, total)
        head = [(names, halves, total, None if seeds is None else [int(s) for s in seeds])]
        if seeds is not None and len(seeds) != total:
            raise ValueError(f"{len(seeds)} seeds for {total} images")
    else:
        tensors, head = None, [None]
    dist.broadcast_object_list(head, src=src, group=group)
    names, halves, total, seed_list = head[0]
    shards = scatter_batch(tensors, device, src=src, group=group)
    kw = _merge_shards(names, halves, shards)
    s, e = shard_ranges(total, world)[rank]
    out = None
    if e > s:
        if seed_list is not None:
            common = dict(common, generator=[torch.Generator().manual_seed(seed_list[i]) for i in range(s, e)])
        res = pipe(**kw, **common)
        out = res.images if hasattr(res, "images") else res[0]
        if not torch.is_tensor(out):
            raise TypeError("sharded_call gathers tensors: use output_type 'uint8', 'pt' or 'latent'")
    # ranks without a request take the trailing shape / dtype of the result from one that has it
    meta = [None] * world
    dist.all_gather_object(meta, None if out is None else (tuple(out.shape[1:]), out.dtype), group=group)
    have = [m for m in meta if m is not None]
    if not have:
        return None
    if out is None:
        out = torch.empty((0,) + have[0][0], dtype=have[0][1], device=device)
    return gather_batch(out.contiguous(), total, dst=src, group=group)
