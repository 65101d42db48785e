"""Variant sharding across the GPUs of one box (SURVEY section 8e).

Every ELBO term is a sum over (replicate, guide) rows and every learnable parameter of the Normal /
MixtureNormal models is per-variant or per-guide, so a contiguous block of variants (with all their
guides, data constants `a0`, `pi_a0`, size factors computed on the WHOLE screen beforehand) is a
self-contained SVI problem: there is NO data-path collective.  The only cross-rank traffic is the ELBO
scalar of each step (summed once, lazily, for the returned loss list) and the final gather of the
parameters.  Noise is indexed by GLOBAL guide / variant ids, so the result does not depend on the world size.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch


def shard_variants(target_lengths, world: int) -> List[Tuple[int, int, int, int]]:
    """Contiguous variant blocks balanced by guide count.

    Returns per rank (variant_begin, variant_end, guide_begin, guide_end); blocks may be empty when there
    are fewer variants than ranks."""
    tl = np.asarray(target_lengths, dtype=np.int64)
    T = len(tl)
    starts = np.concatenate([[0], np.cumsum(tl)])  # guide index where variant v begins
    cuts = [0]
    for r in range(world - 1):
        v0 = cuts[-1]
        left = world - r  # ranks still to be served, this one included
        if T - v0 <= 0:
            cuts.append(T)
            continue
        target = starts[v0] + (starts[T] - starts[v0]) / left
        v1 = int(np.searchsorted(starts, target, side="left"))
        if v1 > v0 + 1 and (target - starts[v1 - 1]) < (starts[v1] - target):
            v1 -= 1  # the nearer boundary
        v1 = max(v1, v0 + 1)  # at least one variant while any remain
        v1 = min(v1, T - min(left - 1, T - v0 - 1))  # leave one for each remaining rank when possible
        cuts.append(v1)
    cuts.append(T)
    return [(int(cuts[r]), int(cuts[r + 1]), int(starts[cuts[r]]), int(starts[cuts[r + 1]])) for r in range(world)]


def shard_guides(n_guides: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous guide blocks of (nearly) equal size: the tiling designs, whose guides have no variant of their own."""
    cuts = [round(r * n_guides / world) for r in range(world + 1)]
    return [(int(cuts[r]), int(cuts[r + 1])) for r in range(world)]


def shard_data(data, rank: int, world: int):
    """This rank's slice of a tensorised screen (+ its global offsets)."""
    if getattr(data, "is_tiling", False):  # guides only: every rank keeps ALL edits (their gradients are summed over the ranks)
        gb, ge = shard_guides(data.n_guides, world)[rank]
        if ge == gb:
            raise ValueError(f"rank {rank} of {world} received no guides")
        sub = data[np.arange(gb, ge)] if (gb, ge) != (0, data.n_guides) else data
        return sub, {"variant_offset": 0, "guide_offset": gb, "n_variants": int(data.n_edits), "n_guides": ge - gb}
    vb, ve, gb, ge = shard_variants(data.target_lengths.numpy(), world)[rank]
    if ge == gb:
        raise ValueError(f"rank {rank} of {world} received no variants")
    sub = data[np.arange(gb, ge)] if (gb, ge) != (0, data.n_guides) else data
    idx = getattr(data, "negctrl_guide_idx", None)
    if idx is not None and sub is not data:  # global guide indices -> this shard's local ones
        idx = np.asarray(idx)
        sub.negctrl_guide_idx = idx[(idx >= gb) & (idx < ge)] - gb
    return sub, {"variant_offset": vb, "guide_offset": gb, "n_variants": ve - vb, "n_guides": ge - gb}


def run_sharded(make_engine: Callable, data, num_steps: int, rank: int, world: int,
                all_reduce_sum: Optional[Callable] = None, all_gather: Optional[Callable] = None,
                log_every: int = 100, all_reduce_min: Optional[Callable] = None) -> Tuple[Dict[str, torch.Tensor], torch.Tensor]:
    """SVI on this rank's shard; returns (global parameters, global loss per step).

    make_engine(sub_data, guide_offset=..., variant_offset=...) -> an engine (.run(n), .losses(), .params(), .gradients(),
    .nonfinite_step(), .snapshot(), .restore()).  `all_reduce_sum(tensor)` / `all_reduce_min(tensor)` /
    `all_gather(tensor) -> list` default to torch.distributed when initialised.  A non-finite step on any rank raises
    run.FitHalted on every rank, at the same step (the smallest over the ranks).
    """
    import torch.distributed as dist

    from .halt import INT32_MAX
    from .run import run_batches

    if all_reduce_sum is None:
        def all_reduce_sum(t):
            if world > 1:
                dist.all_reduce(t)
            return t
    if all_reduce_min is None:
        def all_reduce_min(t):
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return t
    if all_gather is None:
        def all_gather(t):
            if world == 1:
                return [t]
            sizes = [torch.zeros(1, dtype=torch.int64, device=t.device) for _ in range(world)]
            dist.all_gather(sizes, torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device))
            n = int(max(s.item() for s in sizes))
            pad = torch.zeros((n,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
            pad[: t.shape[0]] = t
            outs = [torch.zeros_like(pad) for _ in range(world)]
            dist.all_gather(outs, pad)
            return [o[: int(s.item())] for o, s in zip(outs, sizes)]

    sub, off = shard_data(data, rank, world)
    eng = make_engine(sub, guide_offset=off["guide_offset"], variant_offset=off["variant_offset"])

    def agree(t):  # every rank stops at the first non-finite step of any rank
        word = torch.tensor([INT32_MAX if t is None else t], dtype=torch.int64, device=_device_of(eng))
        t = int(all_reduce_min(word).item())
        return None if t == INT32_MAX else t

    def collect(eng):
        # the per-step ELBO scalars, reduced once for the whole run
        loss = all_reduce_sum(eng.losses().clone().to(_device_of(eng)))
        params = {}
        replicated = getattr(eng, "replicated_params", ())  # tiling: the per-edit parameters, identical on every rank
        for k, v in eng.params().items():
            if v.dim() == 0 or k in replicated:
                params[k] = v
            else:
                params[k] = torch.cat(all_gather(v.contiguous()), dim=0)
        return params, loss.cpu()

    return run_batches(eng, num_steps, log_every, collect=collect, agree=agree, rank=rank, log=False)


def _device_of(eng):
    return getattr(eng, "device", torch.device("cpu"))
