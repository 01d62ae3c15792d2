"""Data-parallel plumbing: one process per GPU, utterances sharded by contiguous slices, no data-path collective.
The only collective of the whole path is the start-up weight broadcast (SURVEY.md §8e): rank 0 loads/builds the
checkpoint, every other rank receives it over NCCL/NVLink (or gloo in the CPU tests)."""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """GPU `rank` of `world` owns utterances [lo, hi): contiguous, sizes differ by at most one."""
    lo = (n_items * rank) // world
    hi = (n_items * (rank + 1)) // world
    return lo, hi


def broadcast_state_dict(sd: Optional[Dict[str, torch.Tensor]], specs: Sequence[Tuple[str, Tuple[int, ...]]], *, src: int = 0,
                         device: Optional[torch.device] = None, group=None) -> Dict[str, torch.Tensor]:
    """Broadcast the fp32 tensors named in `specs` (name, shape) from rank `src` as ONE flat buffer.
    Returns CPU tensors on every rank (the engine copies them to its own device arena)."""
    rank = dist.get_rank(group)
    total = sum(int(torch.Size(s).numel()) for _, s in specs)
    dev = device or torch.device("cpu")
    flat = torch.empty(total, dtype=torch.float32, device=dev)
    if rank == src:
        assert sd is not None
        flat.copy_(torch.cat([sd[k].reshape(-1).to(torch.float32) for k, _ in specs]))
    dist.broadcast(flat, src=src, group=group)
    host = flat.cpu()
    out, off = {}, 0
    for k, s in specs:
        n = int(torch.Size(s).numel())
        out[k] = host[off: off + n].view(s).clone()
        off += n
    return out


def gather_token_lists(local: List[List[int]], group=None) -> List[List[int]]:
    """Optional: collect every rank's token lists on all ranks (tokens are tiny; waveforms stay rank-local)."""
    world = dist.get_world_size(group)
    bucket: List[Optional[List[List[int]]]] = [None] * world
    dist.all_gather_object(bucket, local, group=group)
    return [t for part in bucket for t in (part or [])]


class DataParallelTTS:
    """API-level data parallelism (BASELINE.json configs[3]: batch 512 = 64 per GPU x 8): one process per GPU under
    torchrun, every rank holds a full ``SoproTTS`` on its own device; rank 0 supplies the checkpoint, the other ranks
    receive it in ONE NCCL broadcast over NVLink; ``synthesize_batch`` then runs this rank's contiguous slice of the
    global batch (``shard_range``).  Utterances are independent, so there is no data-path collective; waveforms stay
    rank-local (``gather_token_lists`` exists for the tiny token lists).  Works without torch.distributed (world 1).

    The broadcast lands in device memory and is handed to the engines as host tensors: the C-ABI constructors pack
    their weight arenas on the host (bf16 rounding, epilogue-row interleaving, conv repacking), a one-time ~0.5 GB copy
    at start-up, not part of any timed path."""

    def __init__(self, cfg, state_dict_rank0, tokenizer, mimi_state_dict, *, device, weight_dtype: str = "fp32",
                 text_vocab: Optional[int] = None, mimi_precision: str = "bf16_tc", group=None):
        from .model import SoproTTS
        from .weights import param_specs

        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        sd = state_dict_rank0
        if self.world > 1:
            if text_vocab is None:
                raise ValueError("text_vocab is needed to size the broadcast on ranks that hold no checkpoint")
            specs = [(k, v[0]) for k, v in param_specs(cfg, int(text_vocab)).items()]
            sd = broadcast_state_dict(sd, specs, src=0, device=torch.device(device), group=group)
        self.tts = SoproTTS.from_state_dict(cfg, sd, tokenizer, mimi_state_dict, device=str(device), weight_dtype=weight_dtype,
                                            mimi_precision=mimi_precision)

    def shard(self, n_items: int) -> Tuple[int, int]:
        return shard_range(n_items, self.rank, self.world)

    def synthesize_batch(self, texts: Sequence[str], *, ref=None, refs=None, seeds: Optional[Sequence[int]] = None, **kw):
        """-> (waveforms of THIS rank's utterances, (lo, hi)): texts[lo:hi] of the global batch, with their seeds and,
        for a voice per text, their refs[lo:hi]."""
        if refs is not None and len(refs) != len(texts):
            raise ValueError(f"refs has {len(refs)} entries for {len(texts)} texts")
        lo, hi = self.shard(len(texts))
        if hi <= lo:
            return [], (lo, hi)
        if refs is not None:
            kw["refs"] = list(refs[lo:hi])
        wavs = self.tts.synthesize_batch(list(texts[lo:hi]), ref=ref, seeds=None if seeds is None else list(seeds[lo:hi]), **kw)
        return wavs, (lo, hi)
