"""Batch-sharded data parallelism for the train step: one process per GPU (torch.distributed, NCCL over NVLink),
ONE all-reduce per step on the flat gradient bucket the optimizer already owns (bf16 by default), averaged, followed by
the global-norm clip and the Adam or SGD update on the reduced bucket (identical on every rank).  BatchNorm statistics stay per rank, as
in the reference at the per-GPU batch size.  Scoring shards by sample with a single final gather (gather_scores)."""

import torch
import torch.distributed as dist


def attach(net, bf16_bucket=True, group=None):
    """Synchronise the parameters from rank 0 and hook the gradient all-reduce into net.optimizer.step()."""
    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError('torch.distributed is not initialised')
    world = dist.get_world_size(group)
    with torch.no_grad():
        for t in list(net.parameters()) + list(net.buffers()):
            dist.broadcast(t.data, src=0, group=group)
    from . import engine
    engine.bump_params()          # .data writes do not move autograd's version counters
    engine.bump_stats()
    opt = net.optimizer
    if bf16_bucket and next(net.parameters()).is_cuda:
        opt.grad_dtype = torch.bfloat16

    def allreduce(flat):
        # gloo (CPU tests) has no AVG: sum then scale
        if dist.get_backend(group) == 'nccl':
            dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group)
        else:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
            flat.div_(world)
        return flat

    opt.allreduce = allreduce
    # NCCL collectives can be recorded into a CUDA graph (train_step(graph=True) replays the whole data-parallel step)
    opt.allreduce_capturable = dist.get_backend(group) == 'nccl'
    return net


def shard_range(n, rank=None, world=None):
    """contiguous [start, stop) of n samples owned by `rank` (scoring shards by sample)"""
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    per = (n + world - 1) // world
    return min(n, rank * per), min(n, (rank + 1) * per)


def gather_scores(local, n_total, dst=0, group=None):
    """local: dict name -> (n_local,) tensor.  One gather per call: returns dict name -> (n_total,) on `dst`, None
    elsewhere.  Shards are padded to the common shard length and trimmed after the gather."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    names = sorted(local)
    per = (n_total + world - 1) // world
    dev = local[names[0]].device
    buf = torch.zeros((len(names), per), dtype=torch.float32, device=dev)
    for i, k in enumerate(names):
        buf[i, :local[k].numel()] = local[k].float()
    out = [torch.empty_like(buf) for _ in range(world)] if rank == dst else None
    if dist.get_backend(group) == 'nccl':
        allb = [torch.empty_like(buf) for _ in range(world)]
        dist.all_gather(allb, buf, group=group)
        out = allb if rank == dst else None
    else:
        dist.gather(buf, out, dst=dst, group=group)
    if rank != dst:
        return None
    cat = torch.cat(out, dim=1)[:, :n_total]
    return {k: cat[i] for i, k in enumerate(names)}
