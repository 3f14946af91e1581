"""Data-parallel retrain (SURVEY.md §8f N4): one process per GPU, weights replicated, each rank runs the masked retrain
step on its own shard of the batch and the gradients are averaged with NCCL all-reduces issued INSIDE the backward, one
per layer as soon as that layer's weight gradient is queued, so the NVLink/NVSwitch traffic (203 MB of fp32 gradients
per step) overlaps the backward of the earlier layers.  The reference is single-GPU (src/train.py); this extends its
loop without changing it:

    dist.init_process_group('nccl'); model.cuda(); train_dp.enable(model); broadcast_parameters(model)
    ... the reference's loop: loss = model.loss(model(x_shard), target_shard); loss.backward(); optimizer.step()

BatchNorm uses per-replica batch statistics (no SyncBN): at batch 64 per GPU the statistics are already taken over
64*H*W >= 10,816 values per channel.  Running statistics therefore differ slightly between ranks; average_buffers()
re-synchronises them (call it before evaluation / checkpointing).  Masked weights receive exactly zero gradient on
every rank, so they stay zero after the averaged step.
"""
import torch
import torch.distributed as dist

from .engine_train import train_plan


def enable(model, group=None):
    """Average gradients across the process group inside Darknet's training backward."""
    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("train_dp.enable: torch.distributed is not initialised")
    plan = train_plan(model)
    plan.dp_group = group
    plan.dp_world = dist.get_world_size(group)
    return model


def disable(model):
    plan = model.__dict__.get('_b200_train_plan')
    if plan is not None:
        plan.dp_group, plan.dp_world = None, 1
    return model


def _invalidate_eval_plan(model):
    """The collectives above write through ``.data``: neither the autograd version counters nor the storage addresses
    engine._plan_key watches change, so a compiled eval plan (folded BN, packed weights) would go stale silently."""
    if hasattr(model, '_b200_plan'):
        model._b200_plan = None
        model._b200_watch = None


def broadcast_parameters(model, src=0, group=None):
    """Every rank starts from rank ``src``'s parameters and buffers (masks included)."""
    for t in list(model.parameters()) + list(model.buffers()):
        dist.broadcast(t.data, src=src, group=group)
    _invalidate_eval_plan(model)


def allreduce_gradients(params, group=None):
    """Stand-alone bucketed gradient averaging (one flat all-reduce) for parameters whose gradients were produced
    outside the Darknet autograd node, e.g. by a loss with its own parameters."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    world = dist.get_world_size(group)
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, group=group)
    flat.div_(world)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n


def average_buffers(model, group=None):
    """Average the floating-point buffers (BatchNorm running statistics) over the ranks."""
    world = dist.get_world_size(group)
    for b in model.buffers():
        if b.is_floating_point() and b.dim() == 1:
            dist.all_reduce(b.data, group=group)
            b.data.div_(world)
    _invalidate_eval_plan(model)
