"""Entity-sharded execution of the hot path across the GPUs of one box (SURVEY §8e).

Layout: the entity table ``ent_emb`` [N, d], ``pred_bias`` [N], their gradients and AMSGrad slots are
row-sharded by entity id (contiguous ``EntityShard`` ranges); every other variable is replicated.
Round-1 schedule ("replicated front end"): every rank receives the same global batch, runs the cheap
front end (lookups -> conv -> fused CPG-FC -> q) redundantly and bit-identically, and scores all B
queries against ITS entity rows only.  The exchange steps are the functions below — each is one NCCL
collective on a tiny tensor; dE / dbias / optimizer state of the table never leave their GPU:

  exchange_rows          all-reduce(sum) of the zero-masked [B, d] gather -> every rank has E[e1] exactly
  reduce_scorer_partials all-reduce(sum) of the partial loss (fp64) and the partial dq = G_shard . E_shard
  reduce_sharded_sumsq   all-reduce(sum) of the squared-norm partials of the sharded gradients (global-norm clip)
  reduce_gold_and_counts all-reduce(sum) of the owner-provided gold logits, then of the integer rank counts
  gather_topk            all-gather of the per-shard top-k lists [B, k] (ConvE.predict_topk merges them on device)

"Data-parallel front end" (weak scaling: the global batch grows with the number of GPUs): every rank receives the
global batch [Bg] but runs the front end only on ITS Bg/P rows; the scorer still sees all Bg queries against the
rank's entity rows.  Additional exchange steps:

  scatter_rows           reduce-scatter of the zero-masked [Bg, d] gather -> each rank has E[e1] of its own rows
  gather_batch           all-gather of per-rank [Bl, w] rows (q forward, dx0 backward) into batch order [Bg, w]
  gather_stat_partials   all-gather of the per-chunk batch-norm partial sums -> every rank finalises the statistics of
                         the GLOBAL batch (synchronised batch norm, forward and backward)
  scatter_dq             reduce-scatter of the per-shard partial dq [Bg, d] -> each rank has the summed dq of its rows
  reduce_replicated_grads all-reduce(sum) of the flat bucket of replicated-parameter gradients

All functions work on tensors of any device (NCCL on GPU; gloo on CPU in the unit tests).  A gloo group given CUDA
tensors stages every collective through host memory: that is how the world-2 parity tests run as two processes on ONE
GPU (NCCL refuses two ranks on the same device), so a single-GPU box still exercises the sharded schedule end to end.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


class EntityShard:
    """Contiguous row range [lo, hi) of the entity table owned by ``rank`` (rows per rank rounded up to ``align``)."""

    def __init__(self, num_ent: int, rank: int = 0, world: int = 1, align: int = 128):
        per = -(-num_ent // world)
        per = -(-per // align) * align
        self.num_ent, self.rank, self.world, self.per = num_ent, rank, world, per
        self.lo = min(num_ent, rank * per)
        self.hi = min(num_ent, self.lo + per)

    @property
    def rows(self) -> int:
        return self.hi - self.lo

    def owner(self, ent: int) -> int:
        return int(ent) // self.per

    def __repr__(self):
        return "EntityShard(rank=%d/%d rows=[%d,%d) of %d)" % (self.rank, self.world, self.lo, self.hi, self.num_ent)


def _active(world, group):
    """Whether an exchange step has anything to exchange.  A shard that claims world > 1 without an initialised
    process group would silently keep its non-owned rows at zero, so that is an error (the CPU unit tests that
    exercise one rank's arithmetic in isolation set ALLOW_UNINITIALISED)."""
    if world <= 1:
        return False
    if dist.is_available() and dist.is_initialized():
        return True
    if ALLOW_UNINITIALISED:
        return False
    raise RuntimeError("EntityShard.world = %d but torch.distributed is not initialised: the exchange steps of the "
                       "sharded path cannot run (launch one process per GPU, e.g. with torchrun)" % world)


ALLOW_UNINITIALISED = False


def _staged(t: torch.Tensor, group) -> bool:
    """CUDA tensor on a gloo group: run the collective on a host copy (test path, see the module docstring)."""
    return t.is_cuda and dist.get_backend(group) == "gloo"


class _Done:
    def wait(self):
        return True


def _all_reduce(t, group, async_op=False):
    if _staged(t, group):
        h = t.detach().cpu()
        dist.all_reduce(h, op=dist.ReduceOp.SUM, group=group)
        t.copy_(h)
        return _Done() if async_op else None
    return dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=async_op)


def _reduce_scatter(out, inp, group):
    if _staged(inp, group):
        hi = inp.detach().cpu()
        dist.all_reduce(hi, op=dist.ReduceOp.SUM, group=group)          # gloo has no reduce-scatter: reduce, then slice
        r, n = dist.get_rank(group), out.numel()
        out.copy_(hi.reshape(-1)[r * n:(r + 1) * n].reshape(out.shape))
        return
    dist.reduce_scatter_tensor(out, inp, op=dist.ReduceOp.SUM, group=group)


def _all_gather(out, inp, group):
    if _staged(inp, group):
        hi = inp.detach().cpu().contiguous()
        parts = [torch.empty_like(hi) for _ in range(dist.get_world_size(group))]
        dist.all_gather(parts, hi, group=group)
        out.copy_(torch.cat([p.reshape(-1) for p in parts]).reshape(out.shape))
        return
    dist.all_gather_into_tensor(out, inp, group=group)


def exchange_rows(x_masked: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """x_masked [B, d]: rows owned by this rank filled, all others exactly zero.  Adding zeros is exact in
    fp32, so one all-reduce(sum) delivers every row bit-exactly to every rank."""
    if _active(world, group):
        _all_reduce(x_masked, group)
    return x_masked


def reduce_scorer_partials(loss_sum: torch.Tensor, dq: torch.Tensor, world: int, group=None):
    """Each rank scored all queries against its rows: the loss and dq = sum over shards of G_s . E_s add up."""
    if _active(world, group):
        _all_reduce(loss_sum, group)
        _all_reduce(dq, group)
    return loss_sum, dq


def reduce_sharded_sumsq(sumsq_sharded: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """Squared-norm partials of the row-sharded gradients add across ranks; replicated gradients are identical on
    every rank and are counted once (they are NOT passed here)."""
    if _active(world, group):
        _all_reduce(sumsq_sharded, group)
    return sumsq_sharded


def reduce_gold(gold: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """gold [B]: the logit of e2[b] on the rank that owns entity e2[b], 0 elsewhere."""
    if _active(world, group):
        _all_reduce(gold, group)
    return gold


def reduce_counts(n_greater: torch.Tensor, n_equal: torch.Tensor, world: int, group=None):
    """Integer partial counts add exactly -> ranks are bit-identical for any number of shards."""
    if _active(world, group):
        _all_reduce(n_greater, group)
        _all_reduce(n_equal, group)
    return n_greater, n_equal


def gather_topk(scores: torch.Tensor, ids: torch.Tensor, world: int, group=None, out=None):
    """Per-rank top-k lists [B, k] (scores fp32, global ids int64) -> every rank's lists [P, B, k] in rank order on
    every rank; coper_topk_merge then selects the global top k.  ``out``: optional (scores, ids) [P, B, k] buffers.
    Without an active group the result is this rank's list alone, [1, B, k]."""
    if not _active(world, group):
        if out is None:
            return scores.unsqueeze(0), ids.unsqueeze(0)
        out[0][0].copy_(scores)
        out[1][0].copy_(ids)
        return out[0][:1], out[1][:1]
    P = dist.get_world_size(group)
    if out is None:
        out = (scores.new_empty((P,) + tuple(scores.shape)), ids.new_empty((P,) + tuple(ids.shape)))
    _all_gather(out[0].view((-1,) + tuple(scores.shape[1:])), scores.contiguous(), group)   # [P * B, k] form
    _all_gather(out[1].view((-1,) + tuple(ids.shape[1:])), ids.contiguous(), group)
    return out


# ---- data-parallel front end -------------------------------------------------------------------------------------
def scatter_rows(x_masked_global: torch.Tensor, x_local: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """x_masked_global [Bg, d] as in exchange_rows; rank r receives rows [r*Bl, (r+1)*Bl) summed over the owners
    (bit-exact: one owner, zeros elsewhere)."""
    if _active(world, group):
        _reduce_scatter(x_local, x_masked_global, group)
    else:
        x_local.copy_(x_masked_global)
    return x_local


def gather_batch(x_global: torch.Tensor, x_local: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """Per-rank rows [Bl, w] -> [Bg, w] in batch order on every rank."""
    if _active(world, group):
        _all_gather(x_global, x_local, group)
    else:
        x_global.copy_(x_local)
    return x_global


def gather_stat_partials(all_partials: torch.Tensor, partials: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """partials [nchunk, C, 2] (per-chunk sums the stats kernels write) -> [P*nchunk, C, 2]; the finalise kernels
    then run with nchunk*P chunks and R*P rows: the statistics of the global batch, identical on every rank."""
    if _active(world, group):
        _all_gather(all_partials, partials, group)
    else:
        all_partials.copy_(partials)
    return all_partials


def scatter_dq(dq_partial_global: torch.Tensor, dq_local: torch.Tensor, loss_sum: torch.Tensor, world: int, group=None):
    """Entity-sharded scorer over all Bg queries: partial dq [Bg, d] sums over shards; each rank keeps its rows."""
    if _active(world, group):
        _all_reduce(loss_sum, group)
        _reduce_scatter(dq_local, dq_partial_global, group)
    else:
        dq_local.copy_(dq_partial_global)
    return dq_local


def reduce_replicated_grads(flat: torch.Tensor, world: int, group=None, async_op: bool = False):
    """Gradients of replicated parameters are partial sums over the rank's rows of the batch."""
    if _active(world, group):
        return _all_reduce(flat, group, async_op=async_op)
    return None
