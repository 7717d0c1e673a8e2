"""Batch-sharded sampling across the GPUs of one box (SURVEY.md section 8e).

Every op of the path is per-sample (GroupNorm statistics and attention are per sample; the only
shared quantity is the scalar time), so the latent batch is cut into contiguous slices, one per
rank, each rank integrates its slice with replicated weights and NO per-step communication, and
one all-gather (NCCL over NVLink/NVSwitch on GPUs, gloo in the CPU tests) assembles the result.
The reference has no distributed code at all; this is the B200-native addition.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist

from .sampling import generate_latents_rk4, generate_latents_rk45


def shard_bounds(batch: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced slices: the first ``batch % world_size`` ranks get one extra sample."""
    if batch < 0 or world_size <= 0 or not (0 <= rank < world_size):
        raise ValueError(f"bad shard request batch={batch} world_size={world_size} rank={rank}")
    base, extra = divmod(batch, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_cond(cond, lo: int, hi: int):
    if cond is None:
        return None
    out = dict(cond)
    for key in ("class_cond", "mask_cond"):          # the per-sample conditioning tensors (sampling.py:219-221)
        if out.get(key) is not None:
            out[key] = out[key][lo:hi]
    return out


@torch.no_grad()
def generate_latents_sharded(model, shape, n_steps=50, cond=None, cfg_strength=3.0, source=None,
                             group: Optional[dist.ProcessGroup] = None, gather: bool = True,
                             sampler: Callable = generate_latents_rk4, **sampler_kwargs):
    """Each rank integrates ``source[lo:hi]`` (the same global ``source`` / ``cond`` on every rank,
    e.g. drawn from one seeded generator) and the slices are all-gathered.

    Returns ``(latents, nfe)``; ``latents`` is the full ``[B,...]`` tensor on every rank when
    ``gather`` is true, else this rank's slice.  With uneven slices the gather pads to the
    largest slice and trims.

    RK45 is offered per sample only (``sampler=generate_latents_rk45, per_sample=True``; ``n_steps`` is then
    ignored): every sample has its own step control, so a shard integrates each of its samples as the unsharded
    batch does, and ``nfe`` is the ``[B]`` tensor of per-sample counts, gathered (or sliced) like the latents.  The
    batched RK45 chooses its step size from an error norm over the whole batch, so a shard's own step control would
    integrate each slice differently, and it is refused.
    """
    rk45 = sampler is generate_latents_rk45
    if rk45 and not sampler_kwargs.get("per_sample"):
        raise ValueError("generate_latents_sharded does not offer batched RK45: per-shard step control would change the "
                         "result (use per_sample=True)")

    def run(shape_, cond_, source_, **kw):
        if rk45:                                           # its third positional parameter is cond, not n_steps
            return sampler(model, shape_, cond=cond_, cfg_strength=cfg_strength, source=source_, **kw)
        return sampler(model, shape_, n_steps, cond_, cfg_strength, source=source_, **kw)

    if not dist.is_initialized():
        return run(shape, cond, source, **sampler_kwargs)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    b = shape[0]
    lo, hi = shard_bounds(b, world, rank)
    p = next(model.parameters())
    if source is None:
        raise ValueError("sharded sampling needs an explicit `source` so every rank slices the same noise")
    local_src = source[lo:hi].to(p.device)
    local_shape = (hi - lo,) + tuple(shape[1:])
    # per-sample tensors handed through to the sampler (e.g. init_latents of the img2img branch, sampling.py:104-109)
    # are sliced like the noise; anything else with a leading batch dimension would be silently mis-shaped
    local_kwargs = dict(sampler_kwargs)
    for k, v in sampler_kwargs.items():
        if torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == b:
            local_kwargs[k] = v[lo:hi]
        elif torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] != 1:
            raise ValueError(f"sharded sampling: tensor argument '{k}' has leading dimension {v.shape[0]}, expected the global batch {b}")
    if hi > lo:
        local, nfe = run(local_shape, shard_cond(cond, lo, hi), local_src, **local_kwargs)
    else:
        local, nfe = local_src.clone(), (torch.zeros(0, dtype=torch.int64) if rk45 else n_steps * 4)
    if not gather:
        return local, nfe

    def all_gather(x):
        per = -(-b // world)                               # ceil: padded slice length
        padded = torch.zeros((per,) + tuple(x.shape[1:]), device=x.device, dtype=x.dtype)
        padded[: hi - lo] = x
        full = torch.empty((world * per,) + tuple(x.shape[1:]), device=x.device, dtype=x.dtype)
        dist.all_gather_into_tensor(full, padded, group=group)
        if b % world == 0:
            return full
        pieces = []
        for r in range(world):
            rlo, rhi = shard_bounds(b, world, r)
            pieces.append(full[r * per: r * per + (rhi - rlo)])
        return torch.cat(pieces, dim=0)

    if rk45:                                               # the per-sample counts travel with the latents (NCCL: on the GPU)
        nfe = all_gather(nfe.to(local.device)).cpu()
    return all_gather(local), nfe
