"""Multi-GPU plumbing: clips are independent, so a batch shards across ranks with no intra-step communication.

One process per GPU (torchrun), weights replicated, clip b of the global batch lives on rank b // B_local; the
in-kernel sampler noise is keyed by the GLOBAL clip index, so results do not depend on the world size. The only
collective is one all-gather of the decoded vertex sequences (SURVEY.md §8(e)); the reference has no distributed
code at all. A fan-out call (several sequences per audio clip) shards by audio clip: fanout_shard_range."""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist

from . import lib


def shard_range(n_clips: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, equal-count split (the all-gather needs equal counts): returns (first clip, clip count)."""
    if n_clips % world != 0:
        raise ValueError(f"{n_clips} clips do not split evenly over {world} ranks (pad the batch)")
    per = n_clips // world
    return rank * per, per


def fanout_shard_range(n_audio: int, fanout: int, rank: int, world: int) -> Tuple[Tuple[int, int], Tuple[int, int]]:
    """Shard of a fan-out call (n_audio clips x `fanout` sequences each, sequence a*fanout + k on clip a) by audio clip, so
    that a clip's sequences stay on one rank and its audio is encoded once: returns ((first clip, clip count), (first
    sequence, sequence count)). The first sequence is the rank's `diffusion.clip_index0` (noise keyed by the global sequence
    index), and the gathered (world * count, ...) sequences are in global order."""
    a0, na = shard_range(n_audio, rank, world)
    return (a0, na), (a0 * fanout, na * fanout)


def gather_clips(local: torch.Tensor, group=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """All-gather a per-rank (B_local, ...) tensor into (world * B_local, ...) in rank order."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    local = local.contiguous()
    if out is None:
        out = torch.empty((world * local.shape[0],) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    with lib.nvtx_range("all_gather"):
        dist.all_gather_into_tensor(out.view(-1), local.view(-1), group=group)
    return out


def sample_sharded(run_local: Callable[[int, int], torch.Tensor], n_clips: int, group=None) -> torch.Tensor:
    """run_local(first_clip, count) -> (count, T, V) vertices of this rank's shard; returns all clips on every rank."""
    rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    first, count = shard_range(n_clips, rank, world)
    return gather_clips(run_local(first, count), group)


class OverlappedDecodeGather:
    """Decode the EVQ-VAE output in clip chunks and all-gather chunk k on a side stream while chunk k + 1 decodes, so that
    only the LAST chunk's collective is exposed after the decoder (the reference has no distributed code; SURVEY.md
    section 8(e) names the all-gather of the vertex sequences as the path's only collective).

    Every chunk is decoded straight into this rank's region of the gathered buffer `out` (world, B_local, T, V3) - no
    staging copy - and NCCL's all-gather delivers the peers' chunks into their regions of the same buffer."""

    def __init__(self, group=None, chunks: int = 4):
        self.group = group
        self.chunks = max(1, int(chunks))
        self._stream = None
        self.last_gather_ms = None

    def run(self, decode_chunk: Callable[[int, int, torch.Tensor], None], out: torch.Tensor, time_it: bool = False) -> torch.Tensor:
        """decode_chunk(k0, k1, dst) writes clips [k0, k1) of this rank's shard into dst (k1 - k0, T, V3).
        out: (world, B_local, T, V3), contiguous. Returns out viewed as (world * B_local, T, V3)."""
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        rank = dist.get_rank(self.group) if dist.is_initialized() else 0
        assert out.dim() == 4 and out.shape[0] == world and out.is_contiguous()
        B_local = out.shape[1]
        n = min(self.chunks, B_local) if world > 1 else 1  # a single rank decodes in one pass: nothing to overlap
        bounds = [B_local * i // n for i in range(n + 1)]
        cur = torch.cuda.current_stream()
        if world > 1 and (self._stream is None or self._stream.device != out.device):
            self._stream = torch.cuda.Stream(device=out.device)
        ev0 = ev1 = None
        for i in range(n):
            k0, k1 = bounds[i], bounds[i + 1]
            decode_chunk(k0, k1, out[rank, k0:k1])
            if world == 1:
                continue
            self._stream.wait_stream(cur)  # the chunk is decoded before its all-gather starts; later chunks keep decoding
            with torch.cuda.stream(self._stream):
                if time_it and i == n - 1:
                    ev0 = torch.cuda.Event(enable_timing=True)
                    ev0.record()
                dist.all_gather([out[r, k0:k1] for r in range(world)], out[rank, k0:k1], group=self.group)
                if time_it and i == n - 1:
                    ev1 = torch.cuda.Event(enable_timing=True)
                    ev1.record()
        if world > 1:
            cur.wait_stream(self._stream)
            if ev1 is not None:
                self._timing = (ev0, ev1)  # exposed part: the last chunk's collective (read after a synchronize)
        return out.view(world * B_local, *out.shape[2:])

    def exposed_gather_ms(self):
        t = getattr(self, "_timing", None)
        return None if t is None else t[0].elapsed_time(t[1])
