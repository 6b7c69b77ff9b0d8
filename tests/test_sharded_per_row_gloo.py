"""world_size-2/4 gloo tests of sharded_ge2e_loss(reduction="none") on CPU: each rank's per-utterance losses and the
gradient of sum over ranks of <g_q, L_q>, through the same exchanges as the summed loss (all-gather of C_hat,
reduce-scatter of dC_hat, all-reduce of {dw, db}; no loss all-reduce).  The compute stages are the float64 test double
of test_sharded_gloo.py with the per-row contract of ops.bwd_rows / ops.bwd_finalize (an upstream gradient with one
entry per local utterance row); the result must equal the single-process per-row oracle on the concatenated batch."""
import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_sharded_gloo import TorchStages, _free_port

TOL = 1e-9


class RowStages(TorchStages):
    """TorchStages whose backward stages also take grad_out with one entry per local utterance row."""

    @staticmethod
    def bwd_rows(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, n_local, n_total, spk_offset, M, D, w,
                 b, eps, variant, precision, grad_out, dE_hat=None, row_scale=None):
        if grad_out.numel() == 1:
            return TorchStages.bwd_rows(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, n_local, n_total,
                                        spk_offset, M, D, w, b, eps, variant, precision, grad_out, dE_hat, row_scale)
        assert grad_out.shape == (n_local * M,)
        # the logits' gradient of row r scales with g_r: the scalar stage on a column of upstream gradients
        return TorchStages.bwd_rows(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, n_local, n_total,
                                    spk_offset, M, D, w, b, eps, variant, precision, grad_out[:, None], dE_hat,
                                    row_scale)

    @staticmethod
    def bwd_finalize(E, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, w, b, eps, variant, grad_out,
                     row_scale=None):
        n, M, _ = E.shape
        assert grad_out.numel() in (1, n * M)
        return TorchStages.bwd_finalize(E, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, w, b, eps, variant,
                                        grad_out, row_scale)


def upstream(kind, N, M, world):
    rng = np.random.default_rng(11)
    if kind == "ones":
        return np.ones((N, M))
    if kind == "signed":
        return rng.standard_normal((N, M))
    if kind == "mask":
        return (rng.random((N, M)) > 0.6).astype(np.float64)
    g = rng.standard_normal((N, M))
    g[N // world:2 * N // world] = 0.0          # rank 1 weights none of its rows
    return g


KINDS = ("ones", "signed", "mask", "zero_rank")


def _worker(rank, world, port, N, M, D, variant, fused, q):
    import os
    TorchStages.fused = fused
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle import ge2e_oracle as orc
        from speaker_embedding_ge2e_loss_b200.sharded import shard_bounds, sharded_ge2e_loss
        torch.set_num_threads(1)
        E_all = torch.tensor(orc.make_embeddings(N, M, D, seed=7, kind="clustered"), dtype=torch.float64)
        off, n_local = shard_bounds(N, world, rank)
        out = {}
        for kind in KINDS:
            E = E_all[off:off + n_local].clone().requires_grad_(True)
            w = torch.tensor(10.0, dtype=torch.float64, requires_grad=True)
            b = torch.tensor(-5.0, dtype=torch.float64, requires_grad=True)
            L = sharded_ge2e_loss(E, w, b, 1e-6, variant, "fp32", None, stages=RowStages, reduction="none")
            assert L.shape == (n_local, M)
            g = torch.tensor(upstream(kind, N, M, world)[off:off + n_local])
            L.backward(g)
            out[kind] = (L.detach().numpy(), E.grad.numpy(), w.grad.item(), b.grad.item())
        # the summed loss of the same stages: what reduction="none" with g = 1 must reproduce
        E = E_all[off:off + n_local].clone().requires_grad_(True)
        w = torch.tensor(10.0, dtype=torch.float64, requires_grad=True)
        b = torch.tensor(-5.0, dtype=torch.float64, requires_grad=True)
        loss = sharded_ge2e_loss(E, w, b, 1e-6, variant, "fp32", None, stages=RowStages)
        loss.backward()
        out["sum"] = (loss.item(), E.grad.numpy(), w.grad.item(), b.grad.item())
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(1e-30, np.linalg.norm(np.asarray(b)))


@pytest.mark.parametrize("world,variant,fused", [(2, "softmax", False), (2, "softmax", True), (2, "contrast", False),
                                                 (4, "softmax", True), (4, "contrast", False)])
def test_sharded_per_row_equals_single_process_oracle(world, variant, fused):
    from oracle import ge2e_oracle as orc
    from per_row_oracle import forward_backward_rows
    N, M, D = 8, 3, 16
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, N, M, D, variant, fused, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [o for _, o in sorted((q.get(timeout=180) for _ in range(world)), key=lambda t: t[0])]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    E = orc.make_embeddings(N, M, D, seed=7, kind="clustered")
    for kind in KINDS:
        ref = forward_backward_rows(E, 10.0, -5.0, 1e-6, variant, g=upstream(kind, N, M, world))
        per = np.concatenate([r[kind][0] for r in res])
        dE = np.concatenate([r[kind][1] for r in res])
        assert rel(per, ref["per"]) <= TOL, kind
        assert rel(dE, ref["dE"]) <= TOL, kind
        for r in res:                               # dw, db are global on every rank
            assert abs(r[kind][2] - ref["dw"]) <= TOL * max(1.0, abs(ref["dw"])), kind
            assert abs(r[kind][3] - ref["db"]) <= TOL * max(1.0, abs(ref["db"])), kind
    for r in res:                                   # g = 1 is the summed loss
        s, ones = r["sum"], r["ones"]
        assert rel(ones[1], s[1]) <= TOL
        assert abs(ones[2] - s[2]) <= TOL * max(1.0, abs(s[2])) and abs(ones[3] - s[3]) <= TOL * max(1.0, abs(s[3]))
    total = sum(r["ones"][0].sum() for r in res)
    assert abs(total - res[0]["sum"][0]) <= TOL * abs(res[0]["sum"][0])
