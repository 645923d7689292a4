"""Multi-GPU use of the path (SURVEY.md §8e): environments are independent, so the env batch is
sharded by contiguous index ranges, one process per GPU, with NO data-path collective.  The only
communication is the optional gather of observations / rewards / flags to the learner rank
(and the scatter of actions the other way), through torch.distributed (NCCL on GPUs; gloo in
the CPU tests).

The noise an env sees depends on (seed, GLOBAL env index) only, so results do not depend on the
number of shards (tests/test_gpu_parity.py::test_shkadov_philox_noise_sharding_invariance).
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_range(num_envs, rank, world):
    """Contiguous slice [lo, hi) of global env indices owned by `rank`; sizes differ by at most 1."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, rem = divmod(num_envs, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_sizes(num_envs, world):
    return [shard_range(num_envs, r, world)[1] - shard_range(num_envs, r, world)[0] for r in range(world)]


def make_sharded(name, num_envs, rank=None, world=None, **kwargs):
    """BatchedEnv holding this rank's slice of a global batch of `num_envs` environments."""
    from .batched import BatchedEnv
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    lo, hi = shard_range(num_envs, rank, world)
    from ._capi import PHYSICS
    for k in PHYSICS.get(name, ()):          # per-env physical parameters: this rank's slice
        v = kwargs.get(k)
        if v is not None and np.ndim(v.detach().cpu() if isinstance(v, torch.Tensor) else v) == 1:
            if len(v) != num_envs:
                raise ValueError(f"{k}: expected {num_envs} per-env values, got {len(v)}")
            kwargs[k] = v[lo:hi]
    dev = kwargs.pop("device", torch.cuda.current_device())
    return BatchedEnv(name, batch=hi - lo, device=dev, env_index_base=lo, **kwargs)


def _pad_rows(t, n):
    if t.shape[0] == n:
        return t.contiguous()
    out = torch.zeros((n,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    out[:t.shape[0]] = t
    return out


def gather_to_learner(local, num_envs, dst=0, group=None):
    """Gather per-env rows `local` [n_local, ...] of all ranks on `dst` -> [num_envs, ...] (None elsewhere).
    Uneven shards (sizes differ by at most one row) are padded to the largest shard for the collective."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    sizes = shard_sizes(num_envs, world)
    if local.shape[0] != sizes[rank]:
        raise ValueError(f"rank {rank}: expected {sizes[rank]} rows, got {local.shape[0]}")
    m = max(sizes)
    send = _pad_rows(local, m)
    if rank == dst:
        parts = [torch.empty_like(send) for _ in sizes]
        dist.gather(send, parts, dst=dst, group=group)
        return torch.cat([p[:n] for p, n in zip(parts, sizes)], 0)
    dist.gather(send, None, dst=dst, group=group)
    return None


def all_gather_rows(local, num_envs, group=None):
    """Every rank gets the full [num_envs, ...] tensor (all_gather_into_tensor; padded if uneven)."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    sizes = shard_sizes(num_envs, world)
    m = max(sizes)
    send = _pad_rows(local, m)
    out = torch.empty((world * m,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, send, group=group)
    if len(set(sizes)) == 1:
        return out
    return torch.cat([out[r * m:r * m + n] for r, n in enumerate(sizes)], 0)


def scatter_actions(full, num_envs, src=0, like=None, group=None):
    """Learner -> ranks: `full` [num_envs, ...] on `src` (None elsewhere); returns this rank's rows.
    `like` gives dtype/device/trailing shape on non-source ranks."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    sizes = shard_sizes(num_envs, world)
    m = max(sizes)
    ref = full if rank == src else like
    out = torch.empty((m,) + tuple(ref.shape[1:]), dtype=ref.dtype, device=ref.device)
    if rank == src:
        chunks = [_pad_rows(c, m) for c in torch.split(full, sizes, 0)]
        dist.scatter(out, chunks, src=src, group=group)
    else:
        dist.scatter(out, None, src=src, group=group)
    return out[:sizes[rank]]
