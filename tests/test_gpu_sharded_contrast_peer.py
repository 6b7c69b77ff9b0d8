"""The contrast loss of the speaker-sharded step over peer memory, summed and per-utterance, against the float64 oracle.

  * R ranks emulated on ONE GPU as in test_gpu_sharded_emulated.py: every rank's c_hat_all, dC_local and scalar table
    sit on this GPU between NaN canary rows, the ranks run one after another on one stream, and a device synchronise
    stands where ShardedGE2EPlan(variant="contrast") in peer mode has a cross-rank barrier.
      summed:  prep, publish of the c_hat slice + clear dC_local, barrier, ge2e_b200_fwd_rows,
               ge2e_b200_contrast_bwd_rows_peers, publish of {loss, dw, db}, barrier, finalize.
      "none":  prep, publish, barrier, fwd_rows with per_row, publish of {loss}, barrier; then a backward run twice:
               clear dC_local, barrier, ge2e_b200_contrast_bwd_rows_peers_per_row, publish, barrier, per-row finalize.
    Each case is checked against the oracle (TF32: on the speakers TF32 rounding cannot touch, see
    test_gpu_step.robust_speakers) and against the emulated reduce-scatter path on the same batch, whose forward is the
    same kernel, so the two agree on every row up to the order of the float adds.
  * The inputs both entry points refuse: the code, no launch, no byte of any buffer changed.
  * Two real GPUs (skipped below 2): the plan with peer_memory=True against peer_memory=False.
"""
import math
import os
import subprocess
import sys
import textwrap

import pytest
import torch

from oracle import ge2e_oracle as orc
from per_row_oracle_torch import forward_backward_rows
from test_gpu_sharded_emulated import (ARGUMENT, CONTRAST, EPS, F16, FP32, FP32_SPLIT, SHAPE, TF32, UNSUPPORTED, B, W,
                                       check_rc, ptrs, snapshot, unchanged)
from test_gpu_sharded_per_row import run_shards_rows
from test_gpu_step import DEV, FP32_TOL, TF32_TOL, pkg, robust_speakers, run_shards, trel  # noqa: F401

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class ContrastPeers:
    """Every rank's buffers of a peer-mode ShardedGE2EPlan(variant="contrast") on one GPU.  step(g) is the summed
    step; forward() and backward(g_rows) are the two halves of reduction="none"."""

    def __init__(self, pkg, E, w, b, R, prec):
        self.h = h = pkg.lib()
        N, M, D = E.shape
        self.N, self.M, self.D, self.R, self.prec = N, M, D, R, prec
        nl = self.nl = N // R
        U = nl * M
        dev = E.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.wt, self.bt = (torch.tensor(float(v), **f32) for v in (w, b))
        self.s = torch.cuda.current_stream().cuda_stream
        nan = float("nan")
        # `pad` NaN rows in front of, between and behind the ranks' buffers keep every slice 16-byte aligned
        pad = self.pad = 4 // math.gcd(D, 4)
        assert N % pad == 0 and nl % pad == 0
        self.c_buf = torch.full((R * (N + pad) + pad, D), nan, **f32)
        self.d_buf = torch.full((R * (nl + pad) + pad, D), nan, **f32)
        self.c_all = [self.c_buf[pad + r * (N + pad):pad + r * (N + pad) + N] for r in range(R)]
        self.dC = [self.d_buf[pad + r * (nl + pad):pad + r * (nl + pad) + nl] for r in range(R)]
        self.c_canary = (torch.arange(R + 1, device=dev) * (N + pad))[:, None] + torch.arange(pad, device=dev)
        self.d_canary = (torch.arange(R + 1, device=dev) * (nl + pad))[:, None] + torch.arange(pad, device=dev)
        self.tables = torch.full((R, R, 4), nan, **f32)
        self.nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, CONTRAST, prec)
        self.ranks = [dict(E=E[r * nl:(r + 1) * nl], e_hat=torch.empty((U, D), **f32), cos_diag=torch.empty(U, **f32),
                           accum=torch.empty(4, **f32), row_stat=torch.empty(U, **f32), row_aux=torch.empty(U, **f32),
                           row_kstar=torch.empty(U, dtype=torch.int32, device=dev), per=torch.empty(U, **f32),
                           dE_hat=torch.empty((U, D), **f32), dE=torch.empty((nl, M, D), **f32),
                           ws=torch.zeros(max(self.nb, 1), dtype=torch.uint8, device=dev))
                      for r in range(R)]
        self.owners = ptrs([d.data_ptr() for d in self.dC])

    def _prep_publish(self, clear):
        h, nl, M, D, s = self.h, self.nl, self.M, self.D, self.s
        for r, k in enumerate(self.ranks):
            check_rc(h, h.ge2e_b200_prep(k["E"].data_ptr(), nl, M, D, self.prec, k["e_hat"].data_ptr(),
                                         self.c_all[r][r * nl:].data_ptr(), k["cos_diag"].data_ptr(),
                                         k["accum"].data_ptr(), s), "ge2e_b200_prep")
        for r in range(self.R):
            peers = ptrs([self.c_all[q].data_ptr() + r * nl * D * 4 for q in range(self.R) if q != r])
            check_rc(h, h.ge2e_b200_peer_publish(self.c_all[r][r * nl:].data_ptr(), peers, self.R - 1, 0, nl * D,
                                                 self.dC[r].data_ptr() if clear else None, nl * D if clear else 0, s),
                     "ge2e_b200_peer_publish")
        torch.cuda.synchronize()                                # barrier 1

    def _fwd_rows(self, r, per_row):
        h, k, nl = self.h, self.ranks[r], self.nl
        n0 = h.ge2e_b200_launch_count()
        check_rc(h, h.ge2e_b200_fwd_rows(k["e_hat"].data_ptr(), self.c_all[r].data_ptr(), k["cos_diag"].data_ptr(), nl,
                                         self.N, r * nl, self.M, self.D, self.wt.data_ptr(), self.bt.data_ptr(), EPS,
                                         CONTRAST, self.prec, k["row_stat"].data_ptr(), k["row_kstar"].data_ptr(),
                                         k["row_aux"].data_ptr(), k["accum"].data_ptr(),
                                         k["per"].data_ptr() if per_row else None, None, None, None,
                                         k["ws"].data_ptr() if self.nb else None, self.nb, self.s), "ge2e_b200_fwd_rows")
        assert h.ge2e_b200_launch_count() - n0 == 1

    def _bwd_rows(self, r, g):
        """The peer backward rows call of rank r: g is a device scalar or this rank's [n_local * M] rows.  Returns its
        launches."""
        h, k, nl = self.h, self.ranks[r], self.nl
        fn = h.ge2e_b200_contrast_bwd_rows_peers if g.dim() == 0 else h.ge2e_b200_contrast_bwd_rows_peers_per_row
        n0 = h.ge2e_b200_launch_count()
        check_rc(h, fn(k["e_hat"].data_ptr(), self.c_all[r].data_ptr(), k["cos_diag"].data_ptr(),
                       k["row_stat"].data_ptr(), k["row_kstar"].data_ptr(), nl, self.N, r * nl, self.M, self.D,
                       self.wt.data_ptr(), self.bt.data_ptr(), EPS, self.prec, g.data_ptr(), k["dE_hat"].data_ptr(),
                       k["accum"].data_ptr() + 4, self.owners, self.R, self.s), "contrast_bwd_rows_peers")
        return h.ge2e_b200_launch_count() - n0

    def _publish_scalars(self):
        h = self.h
        for r, k in enumerate(self.ranks):
            rows = ptrs([self.tables[q, r].data_ptr() for q in range(self.R)])
            check_rc(h, h.ge2e_b200_peer_publish(k["accum"].data_ptr(), rows, self.R, 0, 4, None, 0, self.s),
                     "ge2e_b200_peer_publish")
        torch.cuda.synchronize()                                # barrier 2
        for q in range(1, self.R):
            assert torch.equal(self.tables[q], self.tables[0]), f"rank {q}'s scalar table differs from rank 0's"
        return self.tables.sum(dim=1)[0, :3].tolist()

    def _finalize(self, g):
        h, nl, M, D = self.h, self.nl, self.M, self.D
        for r, k in enumerate(self.ranks):
            common = (k["dE_hat"].data_ptr(), self.dC[r].data_ptr(), k["cos_diag"].data_ptr(), k["row_stat"].data_ptr(),
                      k["row_aux"].data_ptr(), None, nl, M, D, self.wt.data_ptr(), self.bt.data_ptr(), EPS, CONTRAST)
            if g.dim() == 0:
                rc = h.ge2e_b200_bwd_finalize(k["E"].data_ptr(), *common, g.data_ptr(), k["dE"].data_ptr(), self.s)
            else:
                rc = h.ge2e_b200_bwd_finalize_per_row_typed(k["E"].data_ptr(), 0, None, *common,
                                                            g[r * nl * M:(r + 1) * nl * M].data_ptr(),
                                                            k["dE"].data_ptr(), 0, self.s)
            check_rc(h, rc, "ge2e_b200_bwd_finalize")
        torch.cuda.synchronize()

    def _exchange_ok(self):
        assert self.c_buf[self.c_canary.reshape(-1)].isnan().all(), "a write left its rank's c_hat_all"
        assert self.d_buf[self.d_canary.reshape(-1)].isnan().all(), "an add left its owner's rows"
        assert not self.c_all[0].isnan().any(), "a slice of c_hat_all was never published"
        for r in range(1, self.R):
            assert unchanged([self.c_all[0]], [self.c_all[r]]), f"rank {r}'s c_hat_all differs from rank 0's"

    def _dE(self):
        return torch.cat([k["dE"].clone() for k in self.ranks])

    def step(self, g=1.0):
        gt = torch.tensor(float(g), device=DEV)
        self._prep_publish(clear=True)
        launches = set()
        for r in range(self.R):
            self._fwd_rows(r, per_row=False)
            launches.add(self._bwd_rows(r, gt))
        torch.cuda.synchronize()
        loss, dw, db = self._publish_scalars()
        self._finalize(gt)
        self._exchange_ok()
        return dict(loss=loss, dE=self._dE(), dw=dw, db=db, launches=launches)

    def forward(self):
        self._prep_publish(clear=False)
        for r in range(self.R):
            self._fwd_rows(r, per_row=True)
        loss = self._publish_scalars()[0]
        self._exchange_ok()
        return dict(loss=loss, per=torch.cat([k["per"] for k in self.ranks]).reshape(self.N, self.M))

    def backward(self, g):
        """g: [N, M] upstream gradient of the whole batch; rank r reads its own rows."""
        gl = g.float().contiguous().reshape(-1)
        for d in self.dC:
            d.zero_()
        torch.cuda.synchronize()                                # barrier 1: every owner's rows are cleared
        launches = {self._bwd_rows(r, gl[r * self.nl * self.M:(r + 1) * self.nl * self.M]) for r in range(self.R)}
        torch.cuda.synchronize()
        loss, dw, db = self._publish_scalars()
        self._finalize(gl)
        self._exchange_ok()
        return dict(loss=loss, dE=self._dE(), dw=dw, db=db, launches=launches)


def check_vs_oracle(got, ref, E, w, tf32):
    """Loss, dE, dw, db (and the per-utterance losses where given); TF32: dE and per on the robust speakers."""
    N, M = E.shape[:2]
    tol = TF32_TOL if tf32 else FP32_TOL
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), (got["loss"], ref["loss"])
    ok = robust_speakers(E, w) if tf32 else torch.ones(N, dtype=torch.bool, device=E.device)
    r = trel(got["dE"][ok], ref["dE"][ok])
    assert r <= tol, r
    if "per" in got:
        assert trel(got["per"][ok], ref["per"].reshape(N, M)[ok]) <= tol
    assert abs(got["dw"] - ref["dw"]) <= (2e-2 if tf32 else tol) * max(1.0, abs(ref["dw"])), (got["dw"], ref["dw"])
    assert abs(got["db"] - ref["db"]) <= 1e-5 * N * M, (got["db"], ref["db"])


def check_vs_reduce_scatter(got, rs):
    """The same forward kernel on the same batch: equal up to the order of the float adds."""
    assert abs(got["loss"] - rs["loss"]) <= 1e-6 * abs(rs["loss"]), (got["loss"], rs["loss"])
    assert trel(got["dE"], rs["dE"]) <= 2e-5, trel(got["dE"], rs["dE"])
    assert abs(got["dw"] - rs["dw"]) <= 1e-4 * max(1.0, abs(rs["dw"])), (got["dw"], rs["dw"])
    assert abs(got["db"] - rs["db"]) <= 1e-4 * max(1.0, abs(rs["db"])), (got["db"], rs["db"])


# (N, M, D, ranks, precision, w, upstream gradient)
STEP_CASES = [
    (256, 6, 128, 2, "fp32", W, 1.0),
    (64, 5, 66, 2, "fp32", W, 1.0),                 # D % 4 != 0: the scalar reductions
    (600, 5, 256, 3, "fp32", W, 1.0),               # n_local = 200: not a multiple of 128
    (600, 5, 256, 3, "tf32", W, 1.0),
    (768, 4, 256, 3, "fp32", -3.0, -1.5),           # negative w, upstream gradient through grad_out
    (2048, 8, 256, 4, "fp32", W, 1.0),
    (2048, 8, 256, 4, "tf32", -3.0, -1.5),
    (1024, 10, 256, 8, "tf32", W, 1.0),             # config 3 on 8 ranks: the tensor-core contrast forward
    (1024, 10, 256, 8, "fp32", W, 1.0),
]


def make_E(N, M, D, R, precision):
    # TF32 cases on random embeddings, whose hardest negatives are mostly well separated (robust_speakers)
    kind = "random" if precision == "tf32" else "clustered"
    return torch.tensor(orc.make_embeddings(N, M, D, seed=N + M + R, kind=kind), device=DEV)


@pytest.mark.parametrize("N,M,D,R,precision,w,g", STEP_CASES)
def test_contrast_peer_step_emulated(pkg, N, M, D, R, precision, w, g):
    from speaker_embedding_ge2e_loss_b200 import _lib
    nl = N // R
    prec = _lib.resolve_precision(precision, nl, N, M, D, CONTRAST)
    assert prec == {"tf32": TF32, "fp32": FP32}[precision]
    if (N, M, D, R) == (1024, 10, 256, 8) and prec == TF32:
        assert pkg.lib().ge2e_b200_path(nl, N, M, D, CONTRAST, TF32) == 1
    E = make_E(N, M, D, R, precision)
    got = ContrastPeers(pkg, E, w, B, R, prec).step(g)
    assert got["launches"] == {1}
    check_vs_oracle(got, forward_backward_rows(E, w, B, EPS, "contrast", g=g), E, w, prec == TF32)
    check_vs_reduce_scatter(got, run_shards(pkg, E, w, B, R, precision, False, variant=CONTRAST, g=g))


# (N, M, D, ranks, precision, w)
ROWS_CASES = [
    (256, 6, 128, 2, "fp32", W),
    (64, 5, 66, 2, "fp32", W),
    (600, 5, 256, 3, "fp32", -3.0),
    (600, 5, 256, 3, "tf32", W),
    (2048, 8, 256, 4, "tf32", W),
    (1024, 10, 256, 8, "tf32", W),
    (1024, 10, 256, 8, "fp32", -3.0),
]


@pytest.mark.parametrize("N,M,D,R,precision,w", ROWS_CASES)
def test_contrast_peer_per_row_emulated(pkg, N, M, D, R, precision, w):
    from speaker_embedding_ge2e_loss_b200 import _lib
    nl = N // R
    prec = _lib.resolve_precision(precision, nl, N, M, D, CONTRAST)
    E = make_E(N, M, D, R, precision)
    run = ContrastPeers(pkg, E, w, B, R, prec)
    fwd = run.forward()
    gen = torch.Generator(device=DEV).manual_seed(N + R)
    signed = torch.randn((N, M), generator=gen, device=DEV)
    signed[torch.rand((N, M), generator=gen, device=DEV) < 0.25] = 0.0       # zeros and negatives
    signed[nl:2 * nl] = 0.0                                                    # and one rank's rows all zero
    for g in (torch.ones((N, M), device=DEV), signed):
        first = run.backward(g)
        second = run.backward(g)                  # repeatable: the backward clears dC_local itself
        assert first["launches"] == second["launches"] == {1}
        assert first["loss"] == fwd["loss"]       # the backward's table carries the forward's loss
        assert trel(second["dE"], first["dE"]) <= 2e-5
        assert abs(second["dw"] - first["dw"]) <= 1e-4 * max(1.0, abs(first["dw"]))
        got = dict(first, per=fwd["per"])
        check_vs_oracle(got, forward_backward_rows(E, w, B, EPS, "contrast", g=g), E, w, prec == TF32)
        rs = run_shards_rows(pkg, E, w, B, R, precision, g, CONTRAST)
        assert trel(fwd["per"], rs["per"]) <= 1e-6
        check_vs_reduce_scatter(got, rs)
    summed = ContrastPeers(pkg, E, w, B, R, prec).step()
    ones = run.backward(torch.ones((N, M), device=DEV))
    check_vs_reduce_scatter(dict(ones, loss=fwd["loss"]), summed)


# ------------------------------------------------------------------ rejected inputs leave no trace
# (id, overrides of the call, expected code); base: N = 1024, M = 6, D = 256, 2 ranks, TF32
REJECTS = [
    ("null_grad", dict(null_grad=True), ARGUMENT),
    ("null_row_kstar", dict(null_kstar=True), ARGUMENT),
    ("one_rank", dict(n_ranks=1), SHAPE),
    ("nine_ranks", dict(n_ranks=9), SHAPE),
    ("n_local_times_ranks_not_n_total", dict(n_local=256), SHAPE),
    ("bad_shape_m1", dict(M_call=1), SHAPE),
    ("null_owner", dict(null_owner=True), ARGUMENT),
    ("misaligned_owner", dict(misalign=4), ARGUMENT),
    ("unaligned_float_owner_scalar_path", dict(misalign=2, D=66, N=64), ARGUMENT),
    ("split_planes", dict(precision=FP32_SPLIT), UNSUPPORTED),
    ("f16_plane", dict(precision=F16), UNSUPPORTED),
    ("unknown_precision", dict(precision=7), ARGUMENT),
]


@pytest.mark.parametrize("per_row", [False, True], ids=["summed", "per_row"])
@pytest.mark.parametrize("case,over,code", REJECTS, ids=[c[0] for c in REJECTS])
def test_contrast_bwd_rows_peers_rejects_without_a_trace(pkg, case, over, code, per_row):
    h = pkg.lib()
    N, M, D, R = over.get("N", 1024), 6, over.get("D", 256), 2
    nl = N // R
    n_local, n_ranks = over.get("n_local", nl), over.get("n_ranks", R)
    U = nl * M
    gen = torch.Generator(device=DEV).manual_seed(7)
    f32 = dict(dtype=torch.float32, device=DEV)
    nan = float("nan")
    e_hat = torch.randn((U, D), generator=gen, **f32)
    c_hat = torch.randn((N, D), generator=gen, **f32)
    cos_diag, row_stat = torch.rand(U, generator=gen, **f32), torch.rand(U, generator=gen, **f32)
    kstar = torch.randint(0, N, (U,), generator=gen, device=DEV, dtype=torch.int32)
    grad = torch.randn(U if per_row else 1, generator=gen, **f32)
    wt, bt = (torch.tensor(v, **f32) for v in (W, B))
    dwdb = torch.full((4,), nan, **f32)
    dE_hat = torch.full((U, D), nan, **f32)
    d_buf = torch.full((n_ranks * (nl + 2) + 2, D), nan, **f32)
    owner = [d_buf[2 + r * (nl + 2):].data_ptr() for r in range(n_ranks)]
    owner[-1] += over.get("misalign", 0)
    if over.get("null_owner"):
        owner[-1] = None
    everything = [e_hat, c_hat, cos_diag, row_stat, kstar, grad, wt, bt, dwdb, dE_hat, d_buf]
    fn = h.ge2e_b200_contrast_bwd_rows_peers_per_row if per_row else h.ge2e_b200_contrast_bwd_rows_peers
    torch.cuda.synchronize()
    before = snapshot(everything)
    n0 = h.ge2e_b200_launch_count()
    rc = fn(e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(), row_stat.data_ptr(),
            None if over.get("null_kstar") else kstar.data_ptr(), n_local, N, 0, over.get("M_call", M), D,
            wt.data_ptr(), bt.data_ptr(), EPS, over.get("precision", TF32),
            None if over.get("null_grad") else grad.data_ptr(), dE_hat.data_ptr(), dwdb.data_ptr(), ptrs(owner),
            n_ranks, torch.cuda.current_stream().cuda_stream)
    launched = h.ge2e_b200_launch_count() - n0
    torch.cuda.synchronize()
    assert rc == code, (rc, h.ge2e_b200_strerror(rc).decode())
    assert launched == 0, f"a refused call launched {launched} kernel(s)"
    assert unchanged(before, everything), "a refused call wrote into a buffer"


# ------------------------------------------------------------------ two real GPUs: the plan's own peer-mode wiring
PEER_CHILD = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, %r)
    import torch, torch.distributed as dist
    from speaker_embedding_ge2e_loss_b200 import ShardedGE2EPlan
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    N, M, D = 600, 5, 256                       # n_local = 300: not a multiple of 128
    nl, off = N // world, rank * (N // world)
    gen = torch.Generator().manual_seed(5)
    E_all = torch.nn.functional.normalize(torch.randn(N, M, D, generator=gen), dim=-1).to(dev)
    g_all = torch.randn(N, M, generator=gen).to(dev)
    shard = E_all[off:off + nl].contiguous()
    w = torch.tensor(10.0, device=dev); b = torch.tensor(-5.0, device=dev)
    def rel(a, r):
        return ((a.double() - r.double()).norm() / r.double().norm().clamp_min(1e-30)).item()
    def agree(p, q, what):
        assert rel(p.dE, q.dE) <= 2e-5, (what, rel(p.dE, q.dE))
        for x, y in ((p.loss, q.loss), (p.dw, q.dw), (p.db, q.db)):
            assert abs(x.item() - y.item()) <= 1e-4 * max(1.0, abs(y.item())), (what, x.item(), y.item())
    for precision in ("fp32", "tf32"):
        peer = ShardedGE2EPlan(nl, N, off, M, D, "contrast", precision, device=dev, peer_memory=True)
        nccl = ShardedGE2EPlan(nl, N, off, M, D, "contrast", precision, device=dev, peer_memory=False)
        auto = ShardedGE2EPlan(nl, N, off, M, D, "contrast", precision, device=dev)
        assert peer.peer and auto.peer and not nccl.peer, auto.peer_error
        for _ in range(2):
            peer.step(shard, w, b); nccl.step(shard, w, b)
        torch.cuda.synchronize()
        agree(peer, nccl, ("sum", precision))
        g = peer.capture(shard, w, b)
        g.replay(); torch.cuda.synchronize()
        agree(peer, nccl, ("sum graph", precision))
        del g
        peer = ShardedGE2EPlan(nl, N, off, M, D, "contrast", precision, device=dev, peer_memory=True, reduction="none")
        nccl = ShardedGE2EPlan(nl, N, off, M, D, "contrast", precision, device=dev, peer_memory=False, reduction="none")
        assert peer.peer and not nccl.peer
        for p in (peer, nccl):
            p.grad_rows.copy_(g_all[off:off + nl])
            p.step(shard, w, b, backward=False); p.backward(shard, w, b)
        peer.backward(shard, w, b)
        torch.cuda.synchronize()
        assert rel(peer.per_row, nccl.per_row) <= 1e-6
        agree(peer, nccl, ("none", precision))
        fwd = peer.capture(shard, w, b, backward=False)
        bwd = peer.capture_backward(shard, w, b)
        fwd.replay(); bwd.replay(); bwd.replay(); torch.cuda.synchronize()
        agree(peer, nccl, ("none graphs", precision))
        del fwd, bwd
    dist.barrier()
    if rank == 0:
        print("CONTRAST_PEER_PLAN_OK", flush=True)
    torch.cuda.synchronize()
    os._exit(0)
""") % ROOT


def test_contrast_peer_plan_on_two_gpus(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "contrast_peer_child.py"
    script.write_text(PEER_CHILD)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29599", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert "CONTRAST_PEER_PLAN_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
