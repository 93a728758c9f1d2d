"""Multi-GPU plumbing (SURVEY.md §8e): one process per GPU, utterances sharded across ranks, no collective on the
hot path.  torch.distributed is used for exactly two things:

* `load_voice_broadcast` — rank 0 uploads the packed weights, every other rank receives them with an NCCL
  broadcast over NVLink / NVSwitch straight into the engine's HBM buffer (62.6 MB medium, 113 MB high); the
  tensor-core weights are packed by every rank from its own host parse of the voice;
* `synthesize_sharded`   — optional gather of the per-rank results to rank 0 in input order (objects; works on
  gloo too, which is how the CPU test exercises the host logic without a GPU).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import numpy as np

from .host import shard_utterances


class _DeviceBytes:
    """Expose a raw device pointer to torch through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3,
                                         "strides": None}


def load_voice_broadcast(onnx_path: str, device: int, rank: int, src: int = 0):
    """Load a voice on this rank's GPU; only `src` pays the H2D upload, the rest get the weights over NCCL."""
    import torch
    import torch.distributed as dist
    from . import engine
    voice = engine.Voice(onnx_path, device, upload=(rank == src))
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        ptr, nbytes = voice.weight_buffers()
        t = torch.as_tensor(_DeviceBytes(ptr, nbytes), device=torch.device("cuda", device))
        dist.broadcast(t, src=src)
        torch.cuda.synchronize(device)
    return voice


def synthesize_sharded(synth: Callable[[List[Sequence[int]]], List[np.ndarray]], ids_list: Sequence[Sequence[int]],
                       rank: int, world_size: int, gather_to: Optional[int] = 0):
    """Each rank synthesises its length-balanced share; returns all waveforms in input order on `gather_to`
    (None elsewhere), or just this rank's {index: waveform} when gather_to is None."""
    plan = shard_utterances([len(i) for i in ids_list], world_size)
    mine = plan[rank]
    outs = synth([ids_list[i] for i in mine]) if mine else []
    local = {i: o for i, o in zip(mine, outs)}
    if gather_to is None or world_size == 1:
        return [local[i] for i in range(len(ids_list))] if world_size == 1 else local
    import torch.distributed as dist
    gathered = [None] * world_size if rank == gather_to else None
    dist.gather_object(local, gathered, dst=gather_to)
    if rank != gather_to:
        return None
    merged = {}
    for d in gathered:
        merged.update(d)
    return [merged[i] for i in range(len(ids_list))]
