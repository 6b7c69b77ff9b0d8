"""Per-utterance losses on the single-kernel step's shapes: the step cut into a forward launch (through the row losses)
and a backward launch (w G from one upstream gradient per row, then the Jacobians and the fan-out), and
GE2EPlan(reduction="none") on top of it.

Truth is the float64 oracle with an [N, M] upstream gradient (per_row_oracle.py); the fp32-class tolerance 1e-5
(relative norm) as everywhere, plus one rounding of dE for the half types.  The C-ABI cases assert how many kernels
each half launched, so that a dispatch change cannot make them test the staged kernels instead.
"""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from per_row_oracle import forward_backward_rows
from test_gpu_edges import DEV, EPS, FP32_TOL, TF32_TOL, pkg, small_step_mode, trel  # noqa: F401
from test_gpu_per_row_loss import check_vs_oracle, upstreams

pytestmark = pytest.mark.gpu

W, B = 10.0, -5.0
ROUND = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
DT = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}   # ge2e_dtype codes


class Abi:
    """forward_per_row / backward_per_row through the C ABI with buffers of their own, on one shape."""

    def __init__(self, pkg, N, M, D, variant):
        from speaker_embedding_ge2e_loss_b200 import _lib
        self.h, self.N, self.M, self.D = pkg.lib(), N, M, D
        self.v = _lib.VARIANTS[variant]
        self.p = 0                                     # GE2E_FP32: the single-kernel step's precision
        U, f32 = N * M, dict(dtype=torch.float32, device=DEV)
        self.e_hat, self.c_hat = torch.empty(U, D, **f32), torch.empty(N, D, **f32)
        self.cos_diag, self.row_stat, self.row_aux = (torch.empty(U, **f32) for _ in range(3))
        self.kstar = torch.empty(U, dtype=torch.int32, device=DEV)
        self.dE_hat, self.dC_hat = torch.empty(U, D, **f32), torch.empty(N, D, **f32)
        self.ws = {"plain": self.h.ge2e_b200_workspace_bytes(N, N, M, D, self.v, self.p),
                   "step": self.h.ge2e_b200_step_workspace_bytes(N, M, D, self.v, self.p)}
        self.wsbuf = {k: torch.zeros(max(n, 1), dtype=torch.uint8, device=DEV) for k, n in self.ws.items()}
        self.w, self.b = torch.tensor(W, **f32), torch.tensor(B, **f32)

    def forward(self, E, ws="step", row_index=None):
        """(per [N, M], loss, kernels launched)"""
        per = torch.empty(self.N, self.M, dtype=torch.float32, device=DEV)
        self.accum = torch.full((4,), float("nan"), dtype=torch.float32, device=DEV)
        n0 = self.h.ge2e_b200_launch_count()
        rc = self.h.ge2e_b200_forward_per_row_typed(
            E.data_ptr(), DT[E.dtype], None if row_index is None else row_index.data_ptr(), self.N, self.M, self.D,
            self.w.data_ptr(), self.b.data_ptr(), EPS, self.v, self.p, self.e_hat.data_ptr(), self.c_hat.data_ptr(),
            self.cos_diag.data_ptr(), self.row_stat.data_ptr(), self.kstar.data_ptr(), self.row_aux.data_ptr(),
            self.accum.data_ptr(), None, None, per.data_ptr(), self.wsbuf[ws].data_ptr(), self.ws[ws], 0)
        assert rc == 0, rc
        torch.cuda.synchronize()
        return per, self.accum[0].item(), self.h.ge2e_b200_launch_count() - n0

    def backward(self, E, g, ws="step", row_index=None, de_dtype=None):
        """(dE, dw, db, kernels launched) for the last forward and upstream gradient g [N, M]"""
        gr = torch.as_tensor(g, dtype=torch.float32, device=DEV).contiguous()
        dE = torch.full(E.shape, float("nan"), dtype=de_dtype or E.dtype, device=DEV)
        accum = torch.full((4,), float("nan"), dtype=torch.float32, device=DEV)
        n0 = self.h.ge2e_b200_launch_count()
        rc = self.h.ge2e_b200_backward_per_row_typed(
            E.data_ptr(), DT[E.dtype], None if row_index is None else row_index.data_ptr(), self.e_hat.data_ptr(),
            self.c_hat.data_ptr(), self.cos_diag.data_ptr(), self.row_stat.data_ptr(), self.kstar.data_ptr(),
            self.row_aux.data_ptr(), None, self.N, self.M, self.D, self.w.data_ptr(), self.b.data_ptr(), EPS, self.v,
            self.p, gr.data_ptr(), self.dE_hat.data_ptr(), self.dC_hat.data_ptr(), accum.data_ptr(), dE.data_ptr(),
            DT[dE.dtype], self.wsbuf[ws].data_ptr(), self.ws[ws], 0)
        assert rc == 0, rc
        torch.cuda.synchronize()
        return dE, accum[1].item(), accum[2].item(), self.h.ge2e_b200_launch_count() - n0

    def run(self, E, g, ws="step", row_index=None, de_dtype=None):
        per, _, nf = self.forward(E, ws, row_index)
        dE, dw, db, nb = self.backward(E, g, ws, row_index, de_dtype)
        return (per, dE, dw, db), (nf, nb)


def batch(N, M, D, seed, dtype=torch.float32, offset=0):
    """[N, M, D] clustered embeddings; offset > 0: a contiguous view that starts `offset` elements into its storage."""
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=seed, kind="clustered"), device=DEV).to(dtype)
    if offset:
        store = torch.zeros(offset + E.numel(), dtype=dtype, device=DEV)
        store[offset:] = E.reshape(-1)
        E = store[offset:].view(N, M, D)
    return E


def as_result(per, dE, dw, db):
    return per, dE.float(), dw, db


# (N, M, D, E offset): N = 1 (no off-diagonal column), the one-cluster grids, the first N past them, the training and
# test shapes, the envelope, D = 64 / 192, the slow body (D = 100; E at an odd offset), and rows that are not 16-byte
# multiples (D = 66, 101: the centroid gradient goes through the workspace partials, on a cluster grid and beyond)
SHAPES = [(1, 4, 64, 0), (2, 8, 64, 0), (4, 8, 64, 0), (8, 5, 128, 0), (9, 6, 128, 0), (64, 10, 256, 0),
          (128, 16, 256, 0), (16, 7, 64, 0), (16, 6, 192, 0), (12, 5, 100, 0), (10, 6, 128, 1), (6, 5, 66, 0),
          (12, 5, 66, 0), (9, 6, 101, 0)]


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("N,M,D,offset", SHAPES)
def test_split_step_matches_oracle(pkg, N, M, D, offset, variant):
    a = Abi(pkg, N, M, D, variant)
    assert a.ws["step"] > 0, "expected a shape of the single-kernel step"
    E = batch(N, M, D, seed=N * M + D, offset=offset)
    E_np = E.double().cpu().numpy()
    for name, g in upstreams(N, M, seed=N + D).items():
        (per, dE, dw, db), launches = a.run(E, g)
        assert launches == (1, 1), (name, launches)
        ref = forward_backward_rows(E_np, W, B, EPS, variant, g=g)
        check_vs_oracle((per, dE, dw, db), ref, g, FP32_TOL, name)


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("N,M,D", [(4, 8, 64), (64, 10, 256), (12, 5, 100)])
def test_staged_kernels_remain_for_the_plain_workspace_and_mode_0(pkg, N, M, D, variant):
    a = Abi(pkg, N, M, D, variant)
    E = batch(N, M, D, seed=7 * N + D)
    g = upstreams(N, M, seed=3)["zeros_negatives"]
    split, ls = a.run(E, g, "step")
    assert ls == (1, 1)
    plain, lp = a.run(E, g, "plain")
    with small_step_mode(pkg, 0):
        mode0, l0 = a.run(E, g, "step")
    assert lp == l0 and lp[0] > 1 and lp[1] > 1, (lp, l0)
    for other in (plain, mode0):
        assert trel(other[0], split[0]) <= FP32_TOL
        assert trel(other[1], split[1]) <= FP32_TOL
        gs = float(np.sqrt((g * g).sum()))
        assert abs(other[2] - split[2]) <= FP32_TOL * max(1.0, abs(split[2]), gs)
        assert abs(other[3] - split[3]) <= FP32_TOL * max(1.0, abs(split[3]), gs)


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("N,M,D", [(4, 8, 64), (64, 10, 256), (12, 5, 100), (9, 6, 101)])
def test_mixed_forms(pkg, N, M, D, variant):
    """A split forward followed by a staged backward and the reverse: the forward's outputs mean the same thing."""
    a = Abi(pkg, N, M, D, variant)
    E = batch(N, M, D, seed=N + 5 * D)
    E_np = E.double().cpu().numpy()
    g = upstreams(N, M, seed=5)["normal"]
    ref = forward_backward_rows(E_np, W, B, EPS, variant, g=g)
    for fwd_ws, bwd_ws in (("step", "plain"), ("plain", "step")):
        per, _, nf = a.forward(E, fwd_ws)
        dE, dw, db, nb = a.backward(E, g, bwd_ws)
        assert (nf == 1) == (fwd_ws == "step") and (nb == 1) == (bwd_ws == "step")
        check_vs_oracle((per, dE, dw, db), ref, g, FP32_TOL, f"{fwd_ws}->{bwd_ws}")


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
def test_unperm(pkg, variant):
    N, M, D = 64, 10, 256
    a = Abi(pkg, N, M, D, variant)
    E = batch(N, M, D, seed=11)
    perm = torch.randperm(N * M, generator=torch.Generator().manual_seed(2)).to(DEV)
    idx = torch.empty_like(perm)
    idx[perm] = torch.arange(N * M, device=DEV)
    idx = idx.to(torch.int32)
    flat = E.reshape(N * M, D)[perm].contiguous()          # flat[idx].view(N, M, D) == E
    g = upstreams(N, M, seed=9)["zeros_negatives"]
    (per, dE_flat, dw, db), launches = a.run(flat, g, row_index=idx)
    assert launches == (1, 1)
    ref = forward_backward_rows(E.double().cpu().numpy(), W, B, EPS, variant, g=g)
    check_vs_oracle((per, dE_flat[idx.long()].view(N, M, D), dw, db), ref, g, FP32_TOL, "unperm")


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("N,M,D", [(4, 8, 64), (64, 10, 256), (12, 5, 100)])
def test_half_embeddings(pkg, N, M, D, dtype, variant):
    a = Abi(pkg, N, M, D, variant)
    E = batch(N, M, D, seed=N + 13, dtype=dtype)
    E_np = E.double().cpu().numpy()                      # the widened values are the fp32 call's input
    for name, g in upstreams(N, M, seed=4).items():
        (per, dE, dw, db), launches = a.run(E, g)
        assert launches == (1, 1) and dE.dtype == dtype
        ref = forward_backward_rows(E_np, W, B, EPS, variant, g=g)
        check_vs_oracle(as_result(per, dE, dw, db), ref, g, FP32_TOL + ROUND[dtype], name)


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
def test_large_upstream_overflows_fp16_to_inf(pkg, variant):
    """dE is rounded once after the g_r scaling: entries beyond fp16's range become +-inf, never NaN."""
    N, M, D = 64, 10, 256
    a = Abi(pkg, N, M, D, variant)
    E = batch(N, M, D, seed=21, dtype=torch.float16)
    g = upstreams(N, M, seed=6)["normal"] * 1e9
    a.forward(E)
    dE16 = a.backward(E, g)[0]
    a.forward(E)
    dE32 = a.backward(E, g, de_dtype=torch.float32)[0]
    # two runs: the centroid gradient's L2 summation order moves dE32 by fp32 rounding of the largest terms (an
    # absolute error on the small entries), dE16 by up to one fp16 ulp
    assert not torch.isnan(dE16).any()
    inf = torch.isinf(dE16)
    assert inf.any() and (~inf).any()
    assert (dE32[inf].abs() >= 65520.0 * (1 - 1e-5)).all()             # 65520 rounds to inf in fp16
    assert inf[dE32.abs() >= 65520.0 * (1 + 1e-5)].all()
    assert torch.equal(torch.sign(dE16[inf].float()), torch.sign(dE32[inf]))
    fin = ~inf
    a, r = dE16[fin].float(), dE32[fin]
    assert ((a - r).abs() <= 2.0 ** -10 * r.abs() + FP32_TOL * r.abs().max()).all()


# ------------------------------------------------------------------ GE2EPlan(reduction="none")
def plan_none(pkg, N, M, D, precision="fp32", variant="softmax", **kw):
    return pkg.GE2EPlan(N, M, D, variant=variant, precision=precision, device=DEV, reduction="none", **kw)


def params():
    return (torch.tensor(W, device=DEV), torch.tensor(B, device=DEV))


@pytest.mark.parametrize("N,M,D,precision,variant", [
    (4, 8, 64, "fp32", "softmax"), (64, 10, 256, "fp32", "softmax"), (64, 10, 256, "fp32", "contrast"),
    (256, 6, 128, "tf32", "softmax"), (256, 6, 256, "fp32", "softmax"),
])
def test_plan_matches_module(pkg, N, M, D, precision, variant):
    E = batch(N, M, D, seed=N + D)
    g = upstreams(N, M, seed=8)["zeros_negatives"]
    plan = plan_none(pkg, N, M, D, precision, variant)
    plan.grad_rows.copy_(torch.tensor(g, dtype=torch.float32))
    w, b = params()
    plan.step(E, w, b)
    torch.cuda.synchronize()
    crit = pkg.GE2ELoss(None, device=DEV, w=W, b=B, variant=variant, precision=precision, reduction="none")
    Eg = E.clone().requires_grad_(True)
    L = crit(Eg)
    L.backward(torch.as_tensor(g, dtype=torch.float32, device=DEV))
    torch.cuda.synchronize()
    tol = TF32_TOL if plan.path in (1, 3) else FP32_TOL
    assert trel(plan.per_row, L.detach()) <= tol
    assert abs(plan.loss.item() - L.detach().double().sum().item()) <= tol * max(1.0, abs(L.sum().item()))
    assert trel(plan.dE, Eg.grad) <= tol
    gs = float(np.sqrt((g * g).sum()))
    assert abs(plan.dw.item() - crit.w.grad.item()) <= tol * max(1.0, abs(crit.w.grad.item()), gs)
    assert abs(plan.db.item() - crit.b.grad.item()) <= max(tol, 1e-5) * max(1.0, abs(crit.b.grad.item()), gs)


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("N,M,D,precision", [(4, 8, 64, "fp32"), (64, 10, 256, "fp32"), (256, 6, 128, "tf32")])
def test_plan_ones_reproduces_sum(pkg, N, M, D, precision, variant):
    E = batch(N, M, D, seed=3 * N)
    w, b = params()
    none, summed = plan_none(pkg, N, M, D, precision, variant), pkg.GE2EPlan(N, M, D, variant, precision, device=DEV)
    none.step(E, w, b)
    summed.step(E, w, b)
    torch.cuda.synchronize()
    tol = TF32_TOL if summed.path in (1, 3) else FP32_TOL
    assert abs(none.loss.item() - summed.loss.item()) <= tol * max(1.0, abs(summed.loss.item()))
    assert abs(none.per_row.double().sum().item() - summed.loss.item()) <= tol * max(1.0, abs(summed.loss.item()))
    assert trel(none.dE, summed.dE) <= tol
    assert abs(none.dw.item() - summed.dw.item()) <= tol * max(1.0, abs(summed.dw.item()))
    assert abs(none.db.item() - summed.db.item()) <= 1e-5 * N * M


@pytest.mark.parametrize("N,M,D", [(4, 8, 64), (64, 10, 256)])
def test_plan_captured_halves_with_device_mask(pkg, N, M, D):
    """Forward graph, a top-k mask of the per-row losses written into grad_rows on the device, backward graph --
    replayed over rotating batches through one input buffer, against the eager module with the same mask."""
    w, b = params()
    plan = plan_none(pkg, N, M, D)
    batches = [batch(N, M, D, seed=s) for s in (1, 2, 3)]
    Ebuf = batches[0].clone()
    gf = plan.capture(Ebuf, w, b, backward=False)
    gb = plan.capture_backward(Ebuf, w, b)
    assert plan.launches_per_step == 1 and plan.backward_launches == 1
    k = max(1, (N * M) // 4)
    crit = pkg.GE2ELoss(None, device=DEV, w=W, b=B, reduction="none")
    for rep in range(2):
        for Ek in batches:
            Ebuf.copy_(Ek)
            gf.replay()
            flat = plan.per_row.view(-1)
            plan.grad_rows.zero_().view(-1).scatter_(0, torch.topk(flat, k).indices, 1.0)   # the k hardest rows
            gb.replay()
            torch.cuda.synchronize()
            Eg = Ek.clone().requires_grad_(True)
            L = crit(Eg)
            mask = torch.zeros(N * M, device=DEV)
            mask[torch.topk(L.detach().view(-1), k).indices] = 1.0
            L.backward(mask.view(N, M))
            torch.cuda.synchronize()
            assert torch.equal(plan.grad_rows.view(-1), mask)
            assert trel(plan.per_row, L.detach()) <= 1e-6
            assert trel(plan.dE, Eg.grad) <= FP32_TOL
            assert abs(plan.dw.item() - crit.w.grad.item()) <= FP32_TOL * max(1.0, abs(crit.w.grad.item()), k ** 0.5)
            crit.zero_grad()


@pytest.mark.parametrize("N,M,D", [(4, 8, 64), (64, 10, 256)])
def test_plan_launches(pkg, N, M, D):
    w, b = params()
    E = batch(N, M, D, seed=4)
    plan = plan_none(pkg, N, M, D)
    plan.capture(E, w, b)
    assert plan.launches_per_step == 2
    plan_sgd = plan_none(pkg, N, M, D, sgd=(0.01, 3.0))
    w2, b2 = params()
    plan_sgd.capture(E, w2, b2)
    assert plan_sgd.launches_per_step == 3


def test_plan_sgd_tail_matches_torch(pkg):
    N, M, D = 64, 10, 256
    lr, max_norm = 0.01, 0.01                           # small enough that the clip engages
    E = batch(N, M, D, seed=12)
    g = upstreams(N, M, seed=12)["normal"]
    w, b = params()
    plan = plan_none(pkg, N, M, D, sgd=(lr, max_norm))
    plan.grad_rows.copy_(torch.tensor(g, dtype=torch.float32))
    plan.step(E, w, b)
    torch.cuda.synchronize()
    crit = pkg.GE2ELoss(None, device=DEV, w=W, b=B, reduction="none")
    crit(E).backward(torch.as_tensor(g, dtype=torch.float32, device=DEV))
    total = torch.nn.utils.clip_grad_norm_(crit.parameters(), max_norm)
    assert total.item() > max_norm
    with torch.no_grad():
        for p in crit.parameters():
            p -= lr * p.grad
    assert abs(plan.dw.item() - crit.w.grad.item()) <= 1e-5 * max(1.0, abs(crit.w.grad.item()))
    assert abs(plan.db.item() - crit.b.grad.item()) <= 1e-5 * max(1.0, abs(crit.b.grad.item()))
    assert abs(w.item() - crit.w.item()) <= 1e-6 * max(1.0, abs(crit.w.item()))
    assert abs(b.item() - crit.b.item()) <= 1e-6 * max(1.0, abs(crit.b.item()))


def test_plan_bf16(pkg):
    N, M, D = 64, 10, 256
    E = batch(N, M, D, seed=14, dtype=torch.bfloat16)
    g = upstreams(N, M, seed=14)["normal"]
    w, b = params()
    plan = plan_none(pkg, N, M, D, dtype=torch.bfloat16)
    plan.grad_rows.copy_(torch.tensor(g, dtype=torch.float32))
    plan.step(E, w, b)
    torch.cuda.synchronize()
    assert plan.dE.dtype == torch.bfloat16
    ref = forward_backward_rows(E.double().cpu().numpy(), W, B, EPS, "softmax", g=g)
    check_vs_oracle(as_result(plan.per_row, plan.dE, plan.dw.item(), plan.db.item()), ref, g,
                    FP32_TOL + ROUND[torch.bfloat16], "bf16 plan")


def test_plan_backward_before_forward_raises(pkg):
    N, M, D = 4, 8, 64
    w, b = params()
    E = batch(N, M, D, seed=1)
    plan = plan_none(pkg, N, M, D)
    with pytest.raises(RuntimeError, match="before any forward"):
        plan.backward(E, w, b)
    with pytest.raises(RuntimeError, match="reduction='none'"):
        pkg.GE2EPlan(N, M, D, device=DEV).backward(E, w, b)
    plan.step(E, w, b, backward=False)
    with pytest.raises(ValueError, match="last forward"):
        plan.backward(E.clone(), w, b)
    with pytest.raises(ValueError, match="reduction"):
        pkg.GE2EPlan(N, M, D, device=DEV, reduction="mean")
