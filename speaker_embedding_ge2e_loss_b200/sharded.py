"""Speaker-sharded GE2E loss: one process per GPU, speakers block-partitioned across ranks.

Exchange steps (SURVEY.md section 8(e); the reference has no distributed code):
  forward   all-gather of the normalised centroids  C_hat_r[n_local, D] -> C_hat[n_total, D]
            (rows are then complete locally: no cross-rank softmax merge), all-reduce of the loss
  backward  reduce-scatter (sum) of the full-height partial dC_hat[n_total, D] -> owner rows,
            all-reduce of {dw, db}
Every rank returns the same global loss; ``backward`` yields d(global loss)/d(E_local) and the
*global* dw, db on every rank (do not wrap the loss module in DDP: its two scalars are already
reduced here).  With ``reduction="none"`` every rank returns the losses of its own utterance rows
instead (no loss all-reduce); rank q's upstream gradient g_q weights its rows, and the backward
differentiates sum over ranks of <g_q, L_q> with the same exchanges: dE_local includes what the
other ranks' rows send through this rank's centroids, dw / db are global.

The four compute stages are injectable (``stages=``) so the collective plumbing can be tested on
CPU under gloo with a test double; the default is the CUDA C-ABI stages of ``ops.py``.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _lib


class CudaStages:
    """Default stage backend: the C-ABI kernels."""

    @staticmethod
    def prep(E, c_hat_local_out, precision):
        from . import ops
        return ops.prep(E, c_hat_local_out, precision)

    @staticmethod
    def fwd_rows(*a, **k):
        from . import ops
        return ops.fwd_rows(*a, **k)

    @staticmethod
    def bwd_rows(*a, **k):
        from . import ops
        return ops.bwd_rows(*a, **k)

    @staticmethod
    def bwd_finalize(*a, **k):
        from . import ops
        return ops.bwd_finalize(*a, **k)


def shard_bounds(n_total: int, world: int, rank: int):
    """Block partition of speakers: equal shards are required (all-gather / reduce-scatter of
    equal slices).  Returns (spk_offset, n_local)."""
    if n_total % world != 0:
        raise ValueError(f"n_total={n_total} speakers must divide evenly over {world} ranks")
    n_local = n_total // world
    return rank * n_local, n_local


def _inplace_ok(group) -> bool:
    try:
        return dist.get_backend(group) == "nccl"
    except Exception:
        return False


class ShardedGE2EFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, E_local, w, b, eps, variant, precision, group, stages, per_row):
        world = dist.get_world_size(group)
        rank = dist.get_rank(group)
        n_local, M, D = E_local.shape
        n_total = n_local * world
        spk_offset = rank * n_local
        E_local = E_local.contiguous()
        # the normalised centroids are float32 for half-precision embeddings (prep widens E); other dtypes keep E's,
        # so the host-side emulation of the stages can run in float64
        c_dtype = torch.float32 if E_local.dtype in (torch.bfloat16, torch.float16) else E_local.dtype
        c_hat_all = torch.empty((n_total, D), dtype=c_dtype, device=E_local.device)
        mine = c_hat_all[spk_offset:spk_offset + n_local]
        e_hat, cos_diag, accum = stages.prep(E_local, mine, precision)
        # all-gather of the normalised centroids (8.4 MB at N=8192, D=256)
        dist.all_gather_into_tensor(c_hat_all, mine if _inplace_ok(group) else mine.clone(), group=group)
        # want_grad: where the softmax loss runs on tensor cores the forward also leaves the un-normalised
        # dE_hat rows + row_scale (None on every other path) and the backward is the centroid pass alone
        row_stat, row_kstar, row_aux, per, _, dE_hat, row_scale = stages.fwd_rows(
            e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant, precision, accum,
            per_row=per_row, want_grad=any(ctx.needs_input_grad[:3]))
        if per_row:
            loss = per.view(n_local, M)                 # this rank's rows: the objective is summed by the caller
        else:
            loss = accum[0].clone()
            dist.all_reduce(loss, op=dist.ReduceOp.SUM, group=group)
        ctx.save_for_backward(E_local, w, b, e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, dE_hat,
                              row_scale)
        ctx.cfg = (eps, variant, precision, group, stages, n_local, n_total, spk_offset, M, D)
        return loss

    @staticmethod
    def backward(ctx, g):
        E_local, w, b, e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale = ctx.saved_tensors
        eps, variant, precision, group, stages, n_local, n_total, spk_offset, M, D = ctx.cfg
        g = g.contiguous().reshape(-1)                  # the scalar, or one entry per local utterance row
        dE_hat, dC_partial, dwdb = stages.bwd_rows(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux,
                                                   n_local, n_total, spk_offset, M, D, w, b, eps, variant,
                                                   precision, g, dE_hat=dE_hat, row_scale=row_scale)
        dC_local = torch.empty((n_local, D), dtype=dC_partial.dtype, device=dC_partial.device)
        dist.reduce_scatter_tensor(dC_local, dC_partial.contiguous(), op=dist.ReduceOp.SUM, group=group)
        dwdb = dwdb.clone()
        dist.all_reduce(dwdb, op=dist.ReduceOp.SUM, group=group)
        dE = stages.bwd_finalize(E_local, dE_hat, dC_local, cos_diag, row_stat, row_aux, w, b, eps, variant, g,
                                 row_scale=row_scale)
        return dE, dwdb[0], dwdb[1], None, None, None, None, None, None


REDUCTIONS = ("sum", "none")


def sharded_ge2e_loss(E_local, w, b, eps=1e-6, variant="softmax", precision="fp32", group=None,
                      stages=None, *, reduction="sum"):
    """Global GE2E loss over the speakers of all ranks in ``group`` (E_local = this rank's
    [n_local, M, D] block, ranks ordered by speaker index).

    ``reduction``: "sum" (the global loss, the same on every rank) or "none": this rank's per-utterance
    losses L_local[n_local, M] (float32, logical [speaker][utterance] order), differentiable for any upstream
    gradient; the backward gives d(sum over ranks of <g_q, L_q>)/dE_local and the global dw, db."""
    if reduction not in REDUCTIONS:
        raise ValueError(f"reduction must be one of {REDUCTIONS}, got {reduction!r}")
    if E_local.dim() != 3 or E_local.shape[1] < 2:
        raise ValueError(f"embeddings must be [n_local, M>=2, D], got {tuple(E_local.shape)}")
    group = group if group is not None else dist.group.WORLD
    vcode = _lib.VARIANTS[variant]
    if E_local.is_cuda:
        n_local, M, D = E_local.shape
        with torch.cuda.device(E_local.device):
            pcode = _lib.resolve_precision(precision, n_local, n_local * dist.get_world_size(group), M, D, vcode)
    else:       # host-side emulation of the stages (tests): no tensor-core path to resolve to
        pcode = _lib.PRECISIONS[precision]
    return ShardedGE2EFunction.apply(E_local, w, b, float(eps), vcode, pcode, group, stages or CudaStages,
                                     reduction == "none")
