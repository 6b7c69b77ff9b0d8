"""Per-utterance GE2E losses (reduction="none") across speaker shards, against the float64 per-row oracle.

  * Peer memory, R ranks emulated on ONE GPU as in test_gpu_sharded_emulated.py: the call order of
    ShardedGE2EPlan(reduction="none") in peer mode -- prep, publish of the c_hat slice, barrier, rows pass, publish of
    {loss}, barrier; then a backward run twice: clear dC_local, barrier, ge2e_b200_bwd_rows_peers_per_row, publish of
    {loss, dw, db}, barrier, per-row finalize.  A device synchronise stands for every cross-rank barrier.
  * The reduce-scatter path with a per-row upstream gradient (ops.bwd_rows / ops.bwd_finalize, the stages of
    sharded_ge2e_loss): SIMT softmax and contrast at spk_offset > 0, contrast on the TF32 forward, half E.
  * The inputs ge2e_b200_bwd_rows_peers_per_row refuses: the code, no launch, no byte of any buffer changed.
  * World-1 NCCL child processes: ShardedGE2EPlan(reduction="none") against GE2EPlan(reduction="none"), and
    sharded_ge2e_loss(reduction="none") against ge2e_loss(reduction="none").
  * Two real GPUs (skipped below 2): the plan in peer mode against the NCCL plan and the single-GPU plan.
"""
import os
import subprocess
import sys
import textwrap

import pytest
import torch

from oracle import ge2e_oracle as orc
from per_row_oracle_torch import forward_backward_rows
from test_gpu_sharded_emulated import (EPS, F16, FP32, FP32_SPLIT, NAME, SHAPE, SOFTMAX, CONTRAST, TF32, UNSUPPORTED,
                                       ARGUMENT, W, B, check_rc, hybrid_selected, ptrs, run_peers, snapshot, unchanged)
from test_gpu_step import DEV, FP32_TOL, TF32_TOL, check_dev, pkg, robust_speakers, trel  # noqa: F401

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HALF_ROUNDING = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
KINDS = ("ones", "signed", "topk", "zero_rank")


def upstream(kind, per, R, seed=0):
    """[N, M] float32 upstream gradient on the device: ones, signed normal, the top quarter of the per-utterance
    losses (a hard-example mask computed from per_row on the device), or signed normal with rank 1's rows zero."""
    N, M = per.shape
    if kind == "ones":
        return torch.ones_like(per)
    if kind == "topk":
        k = max(1, per.numel() // 4)
        thr = per.reshape(-1).topk(k).values[-1]
        return (per >= thr).float()
    g = torch.randn(per.shape, generator=torch.Generator(device=per.device).manual_seed(seed + 17), device=per.device)
    if kind == "zero_rank":
        nl = N // R
        g[nl:2 * nl] = 0.0
    return g


def check_rows(got, ref, U, tol):
    """check_dev plus the per-utterance losses."""
    check_dev(got, ref, U, tol)
    r = trel(got["per"].reshape(-1), ref["per"].reshape(-1))
    assert r <= tol, r


# ------------------------------------------------------------------ peer-memory step, R ranks on one GPU
class PeerRows:
    """Every rank's buffers of a peer-mode ShardedGE2EPlan(reduction="none") on one GPU, separated by NaN canary rows;
    forward() and backward(g) follow the plan's call order rank by rank."""

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
        self.c_buf = torch.full((R * (N + 1) + 1, D), nan, **f32)
        self.d_buf = torch.full((R * (nl + 1) + 1, D), nan, **f32)
        self.c_all = [self.c_buf[1 + r * (N + 1):1 + r * (N + 1) + N] for r in range(R)]
        self.dC = [self.d_buf[1 + r * (nl + 1):1 + r * (nl + 1) + nl] for r in range(R)]
        self.c_canary = torch.arange(R + 1, device=dev) * (N + 1)
        self.d_canary = torch.arange(R + 1, device=dev) * (nl + 1)
        self.tables = torch.full((R, R, 4), nan, **f32)
        self.nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, prec)
        assert self.nb > 0
        self.ranks = [dict(E=E[r * nl:(r + 1) * nl], e_hat=torch.empty((U, D), **f32), cos_diag=torch.empty(U, **f32),
                           accum=torch.empty(4, **f32), row_stat=torch.empty(U, **f32), row_aux=torch.empty(U, **f32),
                           row_kstar=torch.empty(U, dtype=torch.int32, device=dev), row_scale=torch.empty(U, **f32),
                           per=torch.empty(U, **f32), dE_hat=torch.empty((U, D), **f32),
                           dE=torch.empty((nl, M, D), **f32), ws=torch.zeros(self.nb, dtype=torch.uint8, device=dev))
                      for r in range(R)]
        self.owners = ptrs([d.data_ptr() for d in self.dC])

    def _publish_scalars(self):
        h = self.h
        for r, k in enumerate(self.ranks):
            rows = ptrs([self.tables[q, r].data_ptr() for q in range(self.R)])
            check_rc(h, h.ge2e_b200_peer_publish(k["accum"].data_ptr(), rows, self.R, 0, 4, None, 0, self.s),
                     "ge2e_b200_peer_publish")
        torch.cuda.synchronize()                                # barrier
        for q in range(1, self.R):
            assert torch.equal(self.tables[q], self.tables[0]), f"rank {q}'s scalar table differs from rank 0's"
        return self.tables.sum(dim=1)[0, :3].tolist()

    def _exchange_ok(self):
        assert self.c_buf[self.c_canary].isnan().all() and self.d_buf[self.d_canary].isnan().all(), \
            "a write left its rank's buffer"
        for r in range(1, self.R):
            assert unchanged([self.c_all[0]], [self.c_all[r]]), f"rank {r}'s c_hat_all differs from rank 0's"

    def forward(self):
        h, nl, N, M, D, s = self.h, self.nl, self.N, self.M, self.D, self.s
        for r, k in enumerate(self.ranks):
            check_rc(h, h.ge2e_b200_prep(k["E"].data_ptr(), nl, M, D, self.prec, k["e_hat"].data_ptr(),
                                         self.c_all[r][r * nl:].data_ptr(), k["cos_diag"].data_ptr(),
                                         k["accum"].data_ptr(), s), "ge2e_b200_prep")
        for r in range(self.R):
            peers = ptrs([self.c_all[q].data_ptr() + r * nl * D * 4 for q in range(self.R) if q != r])
            check_rc(h, h.ge2e_b200_peer_publish(self.c_all[r][r * nl:].data_ptr(), peers, self.R - 1, 0, nl * D, None,
                                                 0, s), "ge2e_b200_peer_publish")
        torch.cuda.synchronize()                                # barrier 1
        for r, k in enumerate(self.ranks):
            check_rc(h, h.ge2e_b200_fwd_rows(k["e_hat"].data_ptr(), self.c_all[r].data_ptr(), k["cos_diag"].data_ptr(),
                                             nl, N, r * nl, M, D, self.wt.data_ptr(), self.bt.data_ptr(), EPS, SOFTMAX,
                                             self.prec, k["row_stat"].data_ptr(), k["row_kstar"].data_ptr(),
                                             k["row_aux"].data_ptr(), k["accum"].data_ptr(), k["per"].data_ptr(), None,
                                             k["dE_hat"].data_ptr(), k["row_scale"].data_ptr(), k["ws"].data_ptr(),
                                             self.nb, s), "ge2e_b200_fwd_rows")
            torch.cuda.synchronize()
            assert not k["ws"][:256].any(), f"rank {r}: workspace counters not zero after the rows pass"
        loss = self._publish_scalars()[0]                       # barrier 2
        self._exchange_ok()
        return dict(loss=loss, per=torch.cat([k["per"] for k in self.ranks]).reshape(self.N, M))

    def backward(self, g):
        """g: [N, M] upstream gradient of the whole batch; rank r reads its own rows.  Returns dict(loss, dE, dw, db,
        launches of one ge2e_b200_bwd_rows_peers_per_row call)."""
        h, nl, N, M, D, s = self.h, self.nl, self.N, self.M, self.D, self.s
        gl = [g[r * nl:(r + 1) * nl].contiguous().reshape(-1) for r in range(self.R)]
        for d in self.dC:
            d.zero_()
        torch.cuda.synchronize()                                # barrier 1: every owner's rows are cleared
        launches = set()
        for r, k in enumerate(self.ranks):
            n0 = h.ge2e_b200_launch_count()
            check_rc(h, h.ge2e_b200_bwd_rows_peers_per_row(
                k["e_hat"].data_ptr(), self.c_all[r].data_ptr(), k["cos_diag"].data_ptr(), k["row_stat"].data_ptr(),
                k["row_aux"].data_ptr(), k["row_scale"].data_ptr(), nl, N, r * nl, M, D, self.wt.data_ptr(),
                self.bt.data_ptr(), EPS, SOFTMAX, self.prec, gl[r].data_ptr(), k["dE_hat"].data_ptr(),
                k["accum"].data_ptr() + 4, self.owners, self.R, k["ws"].data_ptr(), self.nb, s),
                "ge2e_b200_bwd_rows_peers_per_row")
            launches.add(h.ge2e_b200_launch_count() - n0)
            torch.cuda.synchronize()
            assert not k["ws"][:256].any(), f"rank {r}: workspace counters not zero after the centroid pass"
        loss, dw, db = self._publish_scalars()                  # barrier 2
        for r, k in enumerate(self.ranks):
            check_rc(h, h.ge2e_b200_bwd_finalize_per_row_typed(
                k["E"].data_ptr(), 0, None, k["dE_hat"].data_ptr(), self.dC[r].data_ptr(), k["cos_diag"].data_ptr(),
                k["row_stat"].data_ptr(), k["row_aux"].data_ptr(), k["row_scale"].data_ptr(), nl, M, D,
                self.wt.data_ptr(), self.bt.data_ptr(), EPS, SOFTMAX, gl[r].data_ptr(), k["dE"].data_ptr(), 0, s),
                "ge2e_b200_bwd_finalize_per_row_typed")
        torch.cuda.synchronize()
        self._exchange_ok()
        assert len(launches) == 1, launches
        return dict(loss=loss, dE=torch.cat([k["dE"].clone() for k in self.ranks]), dw=dw, db=db,
                    launches=launches.pop())


@pytest.fixture(scope="module")
def cfg4_E():
    return torch.tensor(orc.make_embeddings(8192, 16, 256, seed=11, kind="clustered"), device=DEV)


# (N, M, D, ranks, precision, HYB selected, w)
PEER_CASES = [
    (256, 6, 128, 2, "tf32", False, W),             # one owner tile per rank
    (256, 6, 96, 2, "tf32", False, W),              # CTA size 1
    (1024, 6, 256, 2, "fp32", False, W),
    (1024, 6, 256, 2, "tf32", False, -3.0),         # negative w
    (768, 4, 256, 3, "tf32", False, W),
    (2048, 8, 256, 4, "fp32", False, W),
    (2048, 8, 256, 4, "f16", False, W),
    (1024, 10, 256, 8, "tf32", False, W),
    (1024, 10, 256, 8, "fp32", False, W),
    (1024, 10, 256, 8, "f16", False, W),
    (8192, 16, 256, 8, "tf32", True, W),            # config 4 on 8 ranks: HYB + peers
    (8192, 16, 256, 2, "tf32", True, W),            # config 4 on 2 ranks
]


@pytest.mark.parametrize("N,M,D,R,precision,hyb,w", PEER_CASES)
def test_peer_memory_per_row_emulated_vs_oracle(pkg, request, N, M, D, R, precision, hyb, w):
    from speaker_embedding_ge2e_loss_b200 import _lib
    h = pkg.lib()
    nl = N // R
    prec = _lib.resolve_precision(precision, nl, N, M, D, SOFTMAX)
    assert prec == {"tf32": TF32, "fp32": FP32_SPLIT, "f16": F16}[precision]
    if prec == TF32:
        assert hybrid_selected(h, nl, N, M, D) == hyb
    E = (request.getfixturevalue("cfg4_E") if (N, M, D) == (8192, 16, 256) else
         torch.tensor(orc.make_embeddings(N, M, D, seed=N + M + R, kind="clustered"), device=DEV))
    tol = FP32_TOL if prec == FP32_SPLIT else TF32_TOL
    run = PeerRows(pkg, E, w, B, R, prec)
    fwd = run.forward()
    for kind in KINDS:
        g = upstream(kind, fwd["per"], R, seed=N + R)
        ref = forward_backward_rows(E, w, B, EPS, "softmax", g=g)
        first = run.backward(g)
        second = run.backward(g)                            # repeatable: dC_local is cleared by the backward
        assert first["launches"] == 1 + hyb                 # the lone centroid pass (+ the HYB conversion)
        got = dict(first, loss=fwd["loss"], per=fwd["per"])
        assert abs(first["loss"] - fwd["loss"]) == 0.0      # the backward's table carries the forward's loss
        check_rows(got, ref, N * M, tol)
        assert trel(second["dE"], first["dE"]) <= 2e-5, kind   # float atomics: the order of the adds may differ
        assert abs(second["dw"] - first["dw"]) <= 1e-4 * max(1.0, abs(first["dw"]))
        assert abs(second["db"] - first["db"]) <= 1e-4 * max(1.0, abs(first["db"]))
        if kind == "ones":
            summed = run_peers(pkg, E, w, B, R, prec)
            rs = run_shards_rows(pkg, E, w, B, R, NAME[prec], g)
            for other in (summed, rs):
                assert abs(fwd["loss"] - other["loss"]) <= 1e-6 * abs(other["loss"]), (fwd["loss"], other["loss"])
                assert trel(first["dE"], other["dE"]) <= 2e-5, trel(first["dE"], other["dE"])
                assert abs(first["dw"] - other["dw"]) <= 1e-4 * max(1.0, abs(other["dw"]))


# ------------------------------------------------------------------ reduce-scatter path with a per-row gradient
def run_shards_rows(pkg, E, w, b, R, precision, g, variant=SOFTMAX):
    """run_shards of test_gpu_step.py for the per-utterance losses: every shard runs ops.prep / fwd_rows(per_row) /
    bwd_rows / bwd_finalize with its own rows of g[N, M]; the reduce-scatter is the sum of the full-height partials.
    Returns dict(loss, per, dE, dw, db) of the whole batch."""
    from speaker_embedding_ge2e_loss_b200 import _lib, ops
    N, M, D = E.shape
    nl = N // R
    prec = _lib.PRECISIONS[precision]
    dev = E.device
    wt, bt = torch.tensor(float(w), device=dev), torch.tensor(float(b), device=dev)
    c_hat_all = torch.empty((N, D), device=dev)
    st = []
    for r in range(R):
        Er = E[r * nl:(r + 1) * nl].contiguous()
        e_hat, cos_diag, accum = ops.prep(Er, c_hat_all[r * nl:(r + 1) * nl], prec)
        st.append(dict(E=Er, e_hat=e_hat, cos_diag=cos_diag, accum=accum,
                       g=g[r * nl:(r + 1) * nl].float().contiguous().reshape(-1)))
    dC_sum = torch.zeros((N, D), dtype=torch.float64, device=dev)
    loss = dw = db = 0.0
    per = []
    for r, s in enumerate(st):
        off = r * nl
        rs, ks, aux, p, _, dE_hat, row_scale = ops.fwd_rows(s["e_hat"], c_hat_all, s["cos_diag"], nl, N, off, M, D, wt,
                                                            bt, EPS, variant, prec, s["accum"], per_row=True,
                                                            want_grad=True)
        s["dE_hat"], dC_part, dwdb = ops.bwd_rows(s["e_hat"], c_hat_all, s["cos_diag"], rs, ks, aux, nl, N, off, M, D,
                                                  wt, bt, EPS, variant, prec, s["g"], dE_hat=dE_hat,
                                                  row_scale=row_scale)
        s["row_stat"], s["row_aux"], s["row_scale"] = rs, aux, row_scale
        torch.cuda.synchronize()
        dC_sum += dC_part.double()
        loss += s["accum"][0].item()
        dw += dwdb[0].item()
        db += dwdb[1].item()
        per.append(p)
    dE = []
    for r, s in enumerate(st):
        dC_local = dC_sum[r * nl:(r + 1) * nl].float().contiguous()
        dE.append(ops.bwd_finalize(s["E"], s["dE_hat"], dC_local, s["cos_diag"], s["row_stat"], s["row_aux"], wt, bt,
                                   EPS, variant, s["g"], row_scale=s["row_scale"]))
    torch.cuda.synchronize()
    return dict(loss=loss, per=torch.cat(per).reshape(N, M), dE=torch.cat(dE, dim=0), dw=dw, db=db)


@pytest.mark.parametrize("N,M,D,R,variant", [(64, 10, 256, 2, SOFTMAX), (96, 5, 64, 3, SOFTMAX),
                                             (64, 10, 256, 2, CONTRAST), (96, 5, 64, 3, CONTRAST)])
def test_simt_shards_per_row_vs_oracle(pkg, N, M, D, R, variant):
    """SIMT kernels (path 0) at spk_offset > 0 with every kind of upstream gradient."""
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, variant, FP32) == 0
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + R, kind="clustered"), device=DEV)
    name = "softmax" if variant == SOFTMAX else "contrast"
    per = forward_backward_rows(E, W, B, EPS, name)["per"].float()
    for kind in KINDS:
        g = upstream(kind, per, R, seed=N)
        ref = forward_backward_rows(E, W, B, EPS, name, g=g)
        got = run_shards_rows(pkg, E, W, B, R, "fp32", g, variant)
        check_rows(got, ref, N * M, FP32_TOL)


@pytest.mark.parametrize("N,M,D,R,precision", [(1024, 10, 256, 8, "tf32"), (768, 3, 128, 3, "fp32_split"),
                                               (2048, 8, 256, 2, "fp32_split")])
def test_tensor_core_shards_per_row_vs_oracle(pkg, N, M, D, R, precision):
    """The lone per-row centroid pass (RG kernels) into a full-height partial, at spk_offset > 0."""
    from speaker_embedding_ge2e_loss_b200 import _lib
    prec = _lib.PRECISIONS[precision]
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, SOFTMAX, prec) == (1 if prec == TF32 else 2)
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + R + 2, kind="clustered"), device=DEV)
    per = forward_backward_rows(E, W, B, EPS, "softmax")["per"].float()
    for kind in ("signed", "topk"):
        g = upstream(kind, per, R, seed=N)
        ref = forward_backward_rows(E, W, B, EPS, "softmax", g=g)
        got = run_shards_rows(pkg, E, W, B, R, precision, g)
        check_rows(got, ref, N * M, TF32_TOL if prec == TF32 else FP32_TOL)


def test_contrast_shards_per_row_tc_forward_on_robust_rows(pkg):
    """Contrast at config 3 on 8 shards: TF32 tensor-core forward, SIMT gather backward with g_r; dE compared on the
    speakers TF32 rounding cannot touch (see test_gpu_step.robust_speakers)."""
    N, M, D, R = 1024, 10, 256, 8
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, CONTRAST, TF32) == 1
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=4, kind="random"), device=DEV)
    g = upstream("signed", torch.zeros(N, M, device=DEV), R, seed=4)
    ref = forward_backward_rows(E, W, B, EPS, "contrast", g=g)
    got = run_shards_rows(pkg, E, W, B, R, "tf32", g, CONTRAST)
    assert abs(got["loss"] - ref["loss"]) <= TF32_TOL * abs(ref["loss"])
    ok = robust_speakers(E, W)
    assert trel(got["per"][ok], ref["per"][ok].float()) <= TF32_TOL
    err = trel(got["dE"][ok], ref["dE"][ok].float())
    assert err <= TF32_TOL, err


@pytest.mark.parametrize("N,M,D,R,precision,path", [(512, 4, 256, 4, "fp32", 0), (512, 4, 256, 4, "fp32_split", 2),
                                                    (1024, 10, 256, 8, "tf32", 1)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_half_embedding_shards_per_row_vs_oracle(pkg, N, M, D, R, precision, path, dtype):
    """bfloat16 / float16 E through prep_typed and the per-row finalize: dE in E's type, within the precision's class
    plus one rounding to the half type."""
    from speaker_embedding_ge2e_loss_b200 import _lib
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, SOFTMAX, _lib.PRECISIONS[precision]) == path
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + R + 1, kind="clustered"), device=DEV).to(dtype)
    g = upstream("signed", torch.zeros(N, M, device=DEV), R, seed=7)
    ref = forward_backward_rows(E, W, B, EPS, "softmax", g=g)
    got = run_shards_rows(pkg, E, W, B, R, precision, g)
    assert got["dE"].dtype == dtype
    tol = TF32_TOL if path == 1 else FP32_TOL
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"]))
    assert trel(got["per"].reshape(-1), ref["per"].reshape(-1)) <= tol
    r = trel(got["dE"].reshape(-1), ref["dE"].reshape(-1))
    assert r <= tol + HALF_ROUNDING[dtype], r
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"]))
    assert abs(got["db"] - ref["db"]) <= 1e-5 * N * M


# ------------------------------------------------------------------ rejected inputs leave no trace
PEER_REJECTS = [
    ("null_grad_rows", dict(null_grad=True), ARGUMENT),
    ("null_row_scale", dict(null_scale=True), ARGUMENT),
    ("one_rank", dict(n_ranks=1), SHAPE),
    ("nine_ranks", dict(n_ranks=9), SHAPE),
    ("n_local_times_ranks_not_n_total", dict(n_local=256), SHAPE),
    ("owner_rows_not_a_whole_tile", dict(N=1600, M=4, R=8), UNSUPPORTED),
    ("contrast", dict(variant=CONTRAST), UNSUPPORTED),
    ("simt_precision", dict(precision=FP32), UNSUPPORTED),
    ("misaligned_owner", dict(misalign=True), ARGUMENT),
    ("misaligned_owner_hyb", dict(misalign=True, hybrid=1), ARGUMENT),
    ("misaligned_owner_split", dict(misalign=True, precision=FP32_SPLIT), ARGUMENT),
    ("null_owner", dict(null_owner=True), ARGUMENT),
]


@pytest.mark.parametrize("case,over,code", PEER_REJECTS, ids=[c[0] for c in PEER_REJECTS])
def test_bwd_rows_peers_per_row_rejects_without_a_trace(pkg, case, over, code):
    h = pkg.lib()
    N, M, D, R = over.get("N", 1024), over.get("M", 6), over.get("D", 256), over.get("R", 2)
    nl = N // R
    n_local, n_ranks = over.get("n_local", nl), over.get("n_ranks", R)
    variant, prec = over.get("variant", SOFTMAX), over.get("precision", TF32)
    U = nl * M
    hyb_mode = over.get("hybrid", 0)
    assert hybrid_selected(h, nl, N, M, D, hyb_mode) == (hyb_mode == 1)
    h.ge2e_b200_debug_hybrid(hyb_mode)
    try:
        nb = max(h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, TF32), 256)
        gen = torch.Generator(device=DEV).manual_seed(7)
        f32 = dict(dtype=torch.float32, device=DEV)
        nan = float("nan")
        e_hat = torch.randn((U, D), generator=gen, **f32)
        c_hat = torch.randn((N, D), generator=gen, **f32)
        cos_diag = torch.rand(U, generator=gen, **f32)
        row_stat, row_aux, row_scale = (torch.rand(U, generator=gen, **f32) for _ in range(3))
        grad = torch.randn(U, generator=gen, **f32)
        wt, bt = (torch.tensor(v, **f32) for v in (W, B))
        dwdb = torch.full((4,), nan, **f32)
        dE_hat = torch.full((U, D), nan, **f32)
        d_buf = torch.full((n_ranks * (nl + 1) + 1, D), nan, **f32)
        owner = [d_buf[1 + r * (nl + 1):].data_ptr() for r in range(n_ranks)]
        if over.get("misalign"):
            owner[-1] += 4
        if over.get("null_owner"):
            owner[-1] = None
        ws = torch.zeros(nb, dtype=torch.uint8, device=DEV)
        everything = [e_hat, c_hat, cos_diag, row_stat, row_aux, row_scale, grad, wt, bt, dwdb, dE_hat, d_buf, ws]
        torch.cuda.synchronize()
        before = snapshot(everything)
        n0 = h.ge2e_b200_launch_count()
        rc = h.ge2e_b200_bwd_rows_peers_per_row(
            e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(), row_stat.data_ptr(), row_aux.data_ptr(),
            None if over.get("null_scale") else row_scale.data_ptr(), n_local, N, 0, M, D, wt.data_ptr(), bt.data_ptr(),
            EPS, variant, prec, None if over.get("null_grad") else grad.data_ptr(), dE_hat.data_ptr(),
            dwdb.data_ptr(), ptrs(owner), n_ranks, ws.data_ptr(), nb, torch.cuda.current_stream().cuda_stream)
        launched = h.ge2e_b200_launch_count() - n0
        torch.cuda.synchronize()
    finally:
        h.ge2e_b200_debug_hybrid(0)
    assert rc == code, (rc, h.ge2e_b200_strerror(rc).decode())
    assert launched == 0, f"a refused call launched {launched} kernel(s)"
    assert unchanged(before, everything), "a refused call wrote into a buffer"


def test_null_grad_rows_rejected_without_a_trace(pkg):
    """ge2e_b200_bwd_rows_per_row and ge2e_b200_bwd_finalize_per_row_typed with real buffers and no grad_rows."""
    h = pkg.lib()
    N, M, D, R = 1024, 6, 256, 2
    nl, U = N // R, N // R * M
    f32 = dict(dtype=torch.float32, device=DEV)
    gen = torch.Generator(device=DEV).manual_seed(3)
    ins = [torch.randn((U, D), generator=gen, **f32), torch.randn((N, D), generator=gen, **f32)] + \
          [torch.rand(U, generator=gen, **f32) for _ in range(4)]
    e_hat, c_hat, cos_diag, row_stat, row_aux, row_scale = ins
    E = torch.randn((nl, M, D), generator=gen, **f32)
    wt, bt = (torch.tensor(v, **f32) for v in (W, B))
    kst = torch.full((U,), -7, dtype=torch.int32, device=DEV)
    outs = [torch.full((U, D), float("nan"), **f32), torch.full((N * D + 2,), float("nan"), **f32),
            torch.full((nl, M, D), float("nan"), **f32)]
    nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, TF32)
    ws = torch.zeros(nb, dtype=torch.uint8, device=DEV)
    everything = [*ins, E, wt, bt, kst, *outs, ws]
    torch.cuda.synchronize()
    before = snapshot(everything)
    s = torch.cuda.current_stream().cuda_stream
    n0 = h.ge2e_b200_launch_count()
    rc1 = h.ge2e_b200_bwd_rows_per_row(e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(), row_stat.data_ptr(),
                                       kst.data_ptr(), row_aux.data_ptr(), row_scale.data_ptr(), nl, N, nl, M, D,
                                       wt.data_ptr(), bt.data_ptr(), EPS, SOFTMAX, TF32, None, outs[0].data_ptr(),
                                       outs[1].data_ptr(), outs[1].data_ptr() + N * D * 4, ws.data_ptr(), nb, s)
    rc2 = h.ge2e_b200_bwd_finalize_per_row_typed(E.data_ptr(), 0, None, outs[0].data_ptr(), c_hat.data_ptr(),
                                                 cos_diag.data_ptr(), row_stat.data_ptr(), row_aux.data_ptr(),
                                                 row_scale.data_ptr(), nl, M, D, wt.data_ptr(), bt.data_ptr(), EPS,
                                                 SOFTMAX, None, outs[2].data_ptr(), 0, s)
    launched = h.ge2e_b200_launch_count() - n0
    torch.cuda.synchronize()
    assert (rc1, rc2) == (ARGUMENT, ARGUMENT)
    assert launched == 0
    assert unchanged(before, everything)


# ------------------------------------------------------------------ world-1 NCCL child: the plan and the autograd form
CHILD = textwrap.dedent("""
    import os, sys
    import torch, torch.distributed as dist
    sys.path.insert(0, %r)
    from speaker_embedding_ge2e_loss_b200 import GE2EPlan, ShardedGE2EPlan, ge2e_loss
    from speaker_embedding_ge2e_loss_b200.sharded import sharded_ge2e_loss
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29579", RANK="0", WORLD_SIZE="1")
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda:0"))
    dev = torch.device("cuda:0")
    def rel(a, r):
        return ((a.double() - r.double()).norm() / r.double().norm().clamp_min(1e-12)).item()
    def agree(sp, ref, tol, what):
        errs = dict(per=rel(sp.per_row, ref.per_row), loss=rel(sp.loss, ref.loss), dE=rel(sp.dE, ref.dE.view_as(sp.dE)),
                    dw=rel(sp.dw, ref.dw), db=abs(sp.db.item() - ref.db.item()) / max(1.0, abs(ref.db.item())))
        assert all(e <= tol for e in errs.values()), (what, errs)
    for (N, M, D, variant, precision, tol) in [(64, 10, 256, "softmax", "tf32", 2e-3),
                                                (64, 10, 256, "contrast", "fp32", 1e-5),
                                                (48, 8, 128, "softmax", "fp32", 1e-5),
                                                (512, 4, 256, "softmax", "tf32", 2e-3),     # tensor-core rows pass
                                                (512, 4, 256, "softmax", "fp32", 1e-5)]:    # split planes
        gen = torch.Generator().manual_seed(N + M)
        Es = [torch.nn.functional.normalize(torch.randn(N, M, D, generator=gen), dim=-1).to(dev) for _ in range(2)]
        w = torch.tensor(10.0, device=dev); b = torch.tensor(-5.0, device=dev)
        ref = GE2EPlan(N, M, D, variant, precision, device=dev, reduction="none")
        sp = ShardedGE2EPlan(N, N, 0, M, D, variant, precision, device=dev, reduction="none")
        assert sp.per_row.shape == (N, M) and torch.equal(sp.grad_rows, torch.ones(N, M, device=dev))
        # eager: forward, a signed upstream gradient, backward
        g = torch.randn(N, M, generator=gen).to(dev)
        sp.step(Es[0], w, b, backward=False); ref.step(Es[0], w, b, backward=False)
        sp.grad_rows.copy_(g); ref.grad_rows.copy_(g)
        sp.backward(Es[0], w, b); ref.backward(Es[0], w, b); torch.cuda.synchronize()
        agree(sp, ref, tol, ("eager", N, M, D, variant, precision))
        # captured forward graph, a device-side mask from per_row, a captured backward graph replayed twice
        fwd = sp.capture(Es[1], w, b, backward=False)
        bwd = sp.capture_backward(Es[1], w, b)
        fwd.replay()
        sp.grad_rows.copy_(sp.per_row >= sp.per_row.median())       # hard-example mask, on the device
        bwd.replay(); torch.cuda.synchronize()
        first = (sp.dE.clone(), sp.dw.item(), sp.db.item())
        bwd.replay(); torch.cuda.synchronize()
        assert rel(sp.dE, first[0]) <= 1e-5 and abs(sp.dw.item() - first[1]) <= 1e-4 * max(1.0, abs(first[1]))
        ref.step(Es[1], w, b, backward=False); ref.grad_rows.copy_(sp.grad_rows); ref.backward(Es[1], w, b)
        torch.cuda.synchronize()
        agree(sp, ref, tol, ("graphs", N, M, D, variant, precision))
        # errors as GE2EPlan's
        try:
            sp.backward(Es[0], w, b); raise AssertionError("backward() on another E must raise")
        except ValueError:
            pass
        del fwd, bwd
    s = ShardedGE2EPlan(64, 64, 0, 10, 256, "softmax", "tf32", device=dev)
    try:
        s.backward(torch.zeros(64, 10, 256, device=dev), w, b); raise AssertionError("sum plan backward() must raise")
    except RuntimeError:
        pass
    fresh = ShardedGE2EPlan(64, 64, 0, 10, 256, "softmax", "tf32", device=dev, reduction="none")
    try:
        fresh.backward(torch.zeros(64, 10, 256, device=dev), w, b); raise AssertionError("backward() before forward")
    except RuntimeError:
        pass
    # the autograd form against the single-device functional form, same upstream gradient
    for (N, M, D, variant, precision, dtype, tol) in [(64, 10, 256, "softmax", "fp32", torch.float32, 1e-5),
                                                       (64, 10, 256, "contrast", "fp32", torch.float32, 1e-5),
                                                       (512, 4, 256, "softmax", "tf32", torch.float32, 2e-3),
                                                       (512, 4, 256, "softmax", "fp32", torch.bfloat16, 1e-2)]:
        gen = torch.Generator().manual_seed(N + 1)
        E0 = torch.nn.functional.normalize(torch.randn(N, M, D, generator=gen), dim=-1).to(dev, dtype)
        g = torch.randn(N, M, generator=gen).to(dev)
        out = []
        for fn in (lambda E, w, b: sharded_ge2e_loss(E, w, b, 1e-6, variant, precision, reduction="none"),
                   lambda E, w, b: ge2e_loss(E, w, b, 1e-6, variant, precision, reduction="none")):
            E = E0.clone().requires_grad_(True)
            w = torch.tensor(10.0, device=dev, requires_grad=True); b = torch.tensor(-5.0, device=dev, requires_grad=True)
            L = fn(E, w, b)
            assert L.shape == (N, M) and L.dtype == torch.float32
            L.backward(g)
            out.append((L.detach(), E.grad, w.grad, b.grad))
        (L1, dE1, dw1, db1), (L2, dE2, dw2, db2) = out
        assert dE1.dtype == dtype
        errs = dict(L=rel(L1, L2), dE=rel(dE1, dE2), dw=rel(dw1, dw2), db=abs(db1.item() - db2.item()) / max(1.0, abs(db2.item())))
        assert all(e <= tol for e in errs.values()), (N, M, D, variant, precision, dtype, errs)
    print("SHARDED_PER_ROW_OK", flush=True)
    os._exit(0)
""") % ROOT


def test_world1_plan_and_autograd_per_row_match_single_device():
    r = subprocess.run([sys.executable, "-c", CHILD], capture_output=True, text=True, timeout=600)
    assert "SHARDED_PER_ROW_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ------------------------------------------------------------------ two real GPUs: the plan's own peer-mode wiring
PEER_CHILD = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, %r)
    import torch, torch.distributed as dist
    from speaker_embedding_ge2e_loss_b200 import GE2EPlan, ShardedGE2EPlan
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    N, M, D = 1024, 6, 256
    nl, off = N // world, rank * (N // world)
    gen = torch.Generator().manual_seed(3)
    E_all = [torch.nn.functional.normalize(torch.randn(N, M, D, generator=gen), dim=-1).to(dev) for _ in range(2)]
    g_all = torch.randn(N, M, generator=gen).to(dev)
    w = torch.tensor(10.0, device=dev); b = torch.tensor(-5.0, device=dev)
    def rel(a, r):
        return ((a.double() - r.double()).norm() / r.double().norm().clamp_min(1e-30)).item()
    for precision, tol in (("tf32", 2e-5), ("fp32", 5e-6)):
        ref = GE2EPlan(N, M, D, "softmax", precision, device=dev, reduction="none")
        peer = ShardedGE2EPlan(nl, N, off, M, D, "softmax", precision, device=dev, peer_memory=True, reduction="none")
        nccl = ShardedGE2EPlan(nl, N, off, M, D, "softmax", precision, device=dev, peer_memory=False, reduction="none")
        assert peer.peer and not nccl.peer
        ref.grad_rows.copy_(g_all); peer.grad_rows.copy_(g_all[off:off + nl]); nccl.grad_rows.copy_(g_all[off:off + nl])
        for k in (0, 1):
            shard = E_all[k][off:off + nl].contiguous()
            ref.step(E_all[k], w, b); nccl.step(shard, w, b)
            peer.step(shard, w, b, backward=False); peer.backward(shard, w, b); peer.backward(shard, w, b)
            torch.cuda.synchronize()
            for p in (peer, nccl):
                assert rel(p.per_row, ref.per_row[off:off + nl]) <= tol
                assert rel(p.dE, ref.dE[off:off + nl]) <= 4 * tol, (precision, k, rel(p.dE, ref.dE[off:off + nl]))
                assert abs(p.loss.item() - ref.loss.item()) <= 1e-5 * abs(ref.loss.item())
                assert abs(p.dw.item() - ref.dw.item()) <= 1e-4 * max(1.0, abs(ref.dw.item()))
                assert abs(p.db.item() - ref.db.item()) <= 1e-4 * max(1.0, abs(ref.db.item()))
        shard = E_all[0][off:off + nl].contiguous()
        fwd = peer.capture(shard, w, b, backward=False)
        bwd = peer.capture_backward(shard, w, b)
        fwd.replay(); bwd.replay(); bwd.replay(); torch.cuda.synchronize()
        ref.step(E_all[0], w, b); torch.cuda.synchronize()
        assert rel(peer.dE, ref.dE[off:off + nl]) <= 4 * tol and abs(peer.loss.item() - ref.loss.item()) <= 1e-5 * abs(ref.loss.item())
        del fwd, bwd
    dist.barrier()
    if rank == 0:
        print("SHARDED_PER_ROW_PEER_OK", flush=True)
    torch.cuda.synchronize()
    os._exit(0)
""") % ROOT


def test_peer_memory_per_row_plan_on_two_gpus(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "peer_rows_child.py"
    script.write_text(PEER_CHILD)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29589", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert "SHARDED_PER_ROW_PEER_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
