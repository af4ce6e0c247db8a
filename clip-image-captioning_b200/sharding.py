"""Data-parallel sharding of the caption path (SURVEY.md section 8(e)): the image batch is cut into contiguous ranges,
one per rank, weights are replicated, and the only collective is the final all-gather of the caption tokens.

Pure host logic on top of torch.distributed: works with the NCCL backend on GPUs (bench.py, one process per GPU) and
with gloo on CPU tensors (tests/test_sharding_gloo.py)."""
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous range [lo, hi) of rank `rank`: the first n % world ranks own one item more."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank / world size")
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def global_row_ids(n_items: int, rank: int, world: int, device=None) -> torch.Tensor:
    """int64 ids of this rank's items: keys of the per-image Philox streams, so that sampled captions do not depend on
    the number of GPUs."""
    lo, hi = shard_range(n_items, rank, world)
    return torch.arange(lo, hi, dtype=torch.int64, device=device)


def gather_captions(tokens: torch.Tensor, lengths: torch.Tensor, n_items: int, group=None
                    ) -> Tuple[torch.Tensor, torch.Tensor]:
    """All-gather of the per-rank results ([n_local, ...] int32 tokens, [n_local, ...] int32 lengths) into global image
    order.  Ranks may own different counts (ragged tail): shards are padded to the largest one for the collective."""
    if not (dist.is_available() and dist.is_initialized()):
        return tokens, lengths
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    counts = [shard_range(n_items, r, world)[1] - shard_range(n_items, r, world)[0] for r in range(world)]
    if tokens.shape[0] != counts[rank]:
        raise ValueError("rank %d holds %d items, expected %d" % (rank, tokens.shape[0], counts[rank]))
    cap = max(counts)

    def pad(t):
        if t.shape[0] == cap:
            return t.contiguous()
        out = t.new_zeros((cap,) + tuple(t.shape[1:]))
        out[:t.shape[0]] = t
        return out

    tok_parts = [torch.empty((cap,) + tuple(tokens.shape[1:]), dtype=tokens.dtype, device=tokens.device) for _ in range(world)]
    len_parts = [torch.empty((cap,) + tuple(lengths.shape[1:]), dtype=lengths.dtype, device=lengths.device) for _ in range(world)]
    dist.all_gather(tok_parts, pad(tokens), group=group)
    dist.all_gather(len_parts, pad(lengths), group=group)
    tok = torch.cat([p[:c] for p, c in zip(tok_parts, counts)], dim=0)
    ln = torch.cat([p[:c] for p, c in zip(len_parts, counts)], dim=0)
    return tok, ln


def caption_images_sharded(engine, images: torch.Tensor, params, n_items: Optional[int] = None, group=None):
    """`images` holds this rank's shard (see shard_range); returns (tokens, lengths) of ALL images on every rank."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    if n_items is None:
        n_items = images.shape[0] * world
    lo, _ = shard_range(n_items, rank, world)
    # micro-batches sized for the fastest decode path (Engine.micro_batch_for); Philox streams keyed by global image id
    tokens, lengths, _ = engine.caption_dataset(images, params, first_row_id=lo)
    return gather_captions(tokens, lengths, n_items, group)


def caption_images_sharded_continuous(engine, images: torch.Tensor, params, n_items: Optional[int] = None, group=None,
                                      rows: Optional[int] = None):
    """`caption_images_sharded` on Engine.caption_dataset_continuous (greedy / sampling): finished rows take the next
    image of this rank's shard.  Same result up to near-ties, and positions past a caption's length are 0."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    if n_items is None:
        n_items = images.shape[0] * world
    lo, _ = shard_range(n_items, rank, world)
    tokens, lengths, _ = engine.caption_dataset_continuous(images, params, rows=rows, first_row_id=lo)
    return gather_captions(tokens, lengths, n_items, group)
