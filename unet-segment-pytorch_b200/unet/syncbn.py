"""``nn.SyncBatchNorm``: batch statistics over every rank of a process group.

A model converted with ``nn.SyncBatchNorm.convert_sync_batchnorm`` keeps its ``SyncBatchNorm`` children as
parameter and buffer holders like any other BatchNorm.  Such a child synchronises exactly when
``torch.nn.SyncBatchNorm`` does: in training mode, with ``torch.distributed`` initialised and more than one rank
in its ``process_group`` (None: the default group).  Everywhere else it runs the per-rank path unchanged.

Every statistic of the BatchNorm passes is a fixed-order fp64 table ``(rows, k, C)`` of per-block sums that a
finalize kernel folds, whatever its row count.  Synchronising is therefore an in-place ``all_reduce(SUM)`` of that
table between the producing pass and its finalize, with the pixel count summed over the ranks.  Ranks whose
tables have fewer rows (smaller shards) pad them with zero rows to the largest; zero rows change no sum.

The row counts and pixel counts are exchanged on the host.  In eager mode that happens at every call, so ranks
may change their shapes independently.  Inside a CUDA-graph capture no host exchange is possible: the values come
from the eager calls with the same local shape (``BatchShardedTrainer`` runs warm-up steps before it captures).
Collectives go to the process group the modules name; no second communicator is created.
"""
from __future__ import annotations

import torch
import torch.distributed as dist
import torch.nn as nn

_SIZES = {}   # (group, local rows, local count) -> (rows of the largest table, pixel count over the group)


def group_of(bn):
    """The process group ``bn`` synchronises its batch statistics over, or None for per-rank statistics.
    A BatchNorm seen through padding (``layers._BnView``) carries the decision of the module it pads."""
    if hasattr(bn, "sync_group"):
        return bn.sync_group
    if not isinstance(bn, nn.SyncBatchNorm) or not bn.training:
        return None
    if not (dist.is_available() and dist.is_initialized()):
        return None
    group = bn.process_group if bn.process_group is not None else dist.group.WORLD
    return group if dist.get_world_size(group) > 1 else None


def _global_sizes(rows: int, count: int, group, device):
    key = (group, rows, count)
    if torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
        hit = _SIZES.get(key)
        if hit is None:
            raise RuntimeError("SyncBatchNorm: a BatchNorm shape seen for the first time inside a CUDA-graph capture; "
                               "run an eager step with the same shapes first")
        return hit
    t = torch.tensor([rows, count], dtype=torch.int64, device=device)
    dist.all_reduce(t[:1], op=dist.ReduceOp.MAX, group=group)
    dist.all_reduce(t[1:], op=dist.ReduceOp.SUM, group=group)
    hit = _SIZES[key] = tuple(int(v) for v in t.tolist())
    return hit


def exchange(partials: torch.Tensor, count: int, group):
    """(rows, k, C) fp64 sums of this rank and its pixel count -> the same sums over every rank of ``group``
    (padded to the largest row count) and the pixel count over the group."""
    rows = partials.shape[0]
    max_rows, total = _global_sizes(rows, int(count), group, partials.device)
    if max_rows > rows:
        partials = torch.cat([partials, partials.new_zeros((max_rows - rows,) + tuple(partials.shape[1:]))])
    elif not partials.is_contiguous():
        partials = partials.contiguous()
    dist.all_reduce(partials, op=dist.ReduceOp.SUM, group=group)
    return partials, total


def exchanger(group):
    """``exchange`` bound to ``group`` (the callback the backward wrappers of unet.kernels take), or None."""
    if group is None:
        return None
    return lambda partials, count: exchange(partials, count, group)
