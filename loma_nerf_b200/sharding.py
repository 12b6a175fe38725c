"""Ray sharding and gradient exchange for data-parallel training on the GPUs of one box.

The loss of the path is a plain sum over rays (/root/reference/scripts/nerf.py:297-302), so weight
gradients are additive across disjoint ray shards (SURVEY.md 8e): every rank evaluates its shard,
the flat gradient buffer [d_ws | d_bs | loss] is summed over ranks (one all-reduce per step; NCCL
over NVLink on the GPU box, gloo in the CPU tests), and every rank applies the identical optimiser
update, so the replicated weights never diverge.  Rendering needs no exchange: frames / ray blocks
are disjoint.  Nothing here touches the arithmetic; it is plumbing over torch.distributed.
"""
import numpy as np


def shard_bounds(n_items, world_size, rank):
    """Contiguous, near-equal split of n_items over world_size ranks: [lo, hi) of `rank`.
    The first n_items % world_size ranks get one extra item."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad rank/world_size")
    base, extra = divmod(int(n_items), int(world_size))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_rays(batch, world_size, rank, samples_per_ray):
    """Slice a batch dict (numpy arrays or torch tensors) to this rank's rays.  Per-ray arrays
    (leading dim R) are cut at ray boundaries; per-sample arrays (leading dim R*S) at S times them:
    a ray's samples are never split (the compositing scan runs along them)."""
    R = None
    for k in ("target", "dists", "rays_o", "rays_d", "t"):
        if batch.get(k) is not None:
            R = int(batch[k].shape[0])
            break
    if R is None:
        raise ValueError("batch has no per-ray array")
    lo, hi = shard_bounds(R, world_size, rank)
    out = {}
    for k, v in batch.items():
        if v is None or not hasattr(v, "shape") or len(v.shape) == 0:
            out[k] = v
        elif int(v.shape[0]) == R:
            out[k] = v[lo:hi]
        elif int(v.shape[0]) == R * samples_per_ray:
            out[k] = v[lo * samples_per_ray:hi * samples_per_ray]
        else:
            out[k] = v
    return out


def frames_for_rank(n_frames, world_size, rank):
    """Round-robin frame assignment for forward-only rendering (BASELINE config 4)."""
    return list(range(rank, int(n_frames), int(world_size)))


def allreduce_gradients(flat, group=None):
    """Sum the flat [d_ws | d_bs | loss] buffer over the ranks, in place (torch tensor or numpy).
    Returns the same object.  Single-process runs (no initialised process group) are a no-op."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return flat
    if isinstance(flat, np.ndarray):
        t = torch.from_numpy(flat)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return flat
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return flat


def data_parallel_step(trainer, batch, group=None):
    """One data-parallel train step on this rank's shard: gradients, all-reduce, optimiser.

    Every rank applies the gradient of the whole batch.  With a numeric seed that is the sum of the shards' gradients.
    With seed="loss" (train_nerf.py:477) the whole batch's gradient is (sum of the ranks' losses) x (sum of the ranks'
    unit-seed gradients), not the sum of gradients each seeded with its own shard's loss: so the shards are
    differentiated with seed 1, the buffer is summed, and then its gradient part is multiplied by the summed loss
    buf[-1] -- the arithmetic of the fused peer exchange (tc_reduce_kernel)."""
    loss_seed = isinstance(batch.get("seed"), str)   # Trainer: any string seed is the loss
    trainer.grad(**(dict(batch, seed=1.0) if loss_seed else batch))
    trainer.ctx.order_torch_after()       # the collective runs behind torch's current stream
    buf = allreduce_gradients(trainer.grad_buffer(), group)
    if loss_seed:
        buf[:-1] *= buf[-1]
    trainer.ctx.order_after_torch()       # ... and the optimiser behind the collective
    trainer.apply()
