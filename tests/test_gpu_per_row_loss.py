"""Per-utterance GE2E losses (reduction="none") and their per-row upstream gradient, on every kernel path.

Truth is the float64 numpy oracle with an [N, M] upstream gradient (per_row_oracle.py, pinned against torch autograd
in test_oracle_per_row.py).  Tolerance classes as everywhere: relative norm error 1e-5 for the fp32-class paths (SIMT,
split fp16 planes), 2e-3 for TF32 / one fp16 plane.  Every case asserts which path it ran (path_for).
"""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from per_row_oracle import forward_backward_rows
from test_gpu_edges import DEV, EPS, FP32_TOL, TF32_TOL, pkg, trel  # noqa: F401

pytestmark = pytest.mark.gpu

W, B = 10.0, -5.0
ROUND = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}


def upstreams(N, M, seed):
    """The upstream gradients every case runs: normal, zeros and negatives, one-hot (row indexing), all zero."""
    rng = np.random.default_rng(seed)
    mixed = rng.standard_normal((N, M))
    mixed[rng.random((N, M)) < 0.3] = 0.0
    mixed[rng.random((N, M)) < 0.5] *= -3.0
    onehot = np.zeros((N, M))
    onehot[(7 * N) // 11, M - 2] = 1.0
    return {"normal": rng.standard_normal((N, M)), "zeros_negatives": mixed, "onehot": onehot,
            "all_zero": np.zeros((N, M))}


def crit_for(pkg, precision, variant, reduction):
    return pkg.GE2ELoss(None, device=DEV, w=W, b=B, variant=variant, precision=precision, reduction=reduction)


def run_none(crit, E, g, unperm=None, speakers=0):
    """L = crit(E) with reduction="none", L.backward(g): (L, dE, dw, db)."""
    Eg = E.detach().clone().requires_grad_(True)
    crit.w.grad = crit.b.grad = None
    L = crit(Eg) if unperm is None else crit(Eg, unperm=unperm, speakers=speakers)
    L.backward(torch.as_tensor(g, dtype=torch.float32, device=DEV))
    torch.cuda.synchronize()
    return L.detach(), Eg.grad.clone(), crit.w.grad.item(), crit.b.grad.item()


def check_vs_oracle(got, ref, g, tol, name):
    L, dE, dw, db = got
    assert L.dtype == torch.float32 and torch.isfinite(L).all()
    assert trel(L, torch.tensor(ref["per"], device=DEV)) <= tol, name
    assert abs(L.double().sum().item() - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), name
    assert torch.isfinite(dE).all(), name
    if not np.any(g):
        # no upstream gradient: exact zeros (the split planes divide by max |g_r| = 0), never NaN
        assert not dE.any() and dw == 0.0 and db == 0.0, name
        return
    r = trel(dE, torch.tensor(ref["dE"], device=DEV))
    assert r <= tol, (name, r)
    # every row's d L_r / dw, d L_r / db is O(1): the error of the weighted sum grows like |g|, not like |dw|
    gscale = float(np.sqrt((g * g).sum()))
    assert abs(dw - ref["dw"]) <= tol * max(1.0, abs(ref["dw"]), gscale), (name, dw, ref["dw"])
    assert abs(db - ref["db"]) <= max(tol, 1e-5) * max(1.0, abs(ref["db"]), gscale), (name, db, ref["db"])


# (N, M, D, precision, variant, hybrid operand copies, expected path)
CASES = [
    (4, 8, 64, "fp32", "softmax", False, 0),          # SIMT pipeline, reference test size
    (4, 8, 64, "fp32", "contrast", False, 0),
    (64, 10, 256, "fp32", "softmax", False, 0),       # ... reference training size
    (64, 10, 256, "fp32", "contrast", False, 0),
    (160, 5, 96, "fp32", "softmax", False, 0),        # N >= 129 on SIMT: D not covered by the split planes
    (256, 6, 128, "tf32", "softmax", False, 1),       # tensor-core step, pass 2 alone
    (256, 6, 128, "tf32", "softmax", True, 1),        # ... MMA1 on fp16 operand copies
    (256, 6, 256, "fp32", "softmax", False, 2),       # split fp16 planes
    (256, 6, 256, "f16", "softmax", False, 3),        # one fp16 plane
    (256, 6, 128, "tf32", "contrast", False, 1),      # tensor-core forward + SIMT gather backward
    (1024, 10, 256, "fp32", "softmax", False, 2),     # config 3
    (1024, 10, 256, "tf32", "softmax", False, 1),
]


class hybrid_mode:
    """ge2e_b200_debug_hybrid(1) for a block; the eager plans cache their workspace size per shape, so they are
    dropped on entry and exit."""

    def __init__(self, pkg, on):
        self.pkg, self.on = pkg, on

    def __enter__(self):
        if self.on:
            from speaker_embedding_ge2e_loss_b200 import ops
            ops._EAGER_PLANS.clear()
            self.pkg.lib().ge2e_b200_debug_hybrid(1)

    def __exit__(self, *a):
        if self.on:
            from speaker_embedding_ge2e_loss_b200 import ops
            self.pkg.lib().ge2e_b200_debug_hybrid(0)
            ops._EAGER_PLANS.clear()


@pytest.mark.parametrize("N,M,D,precision,variant,hybrid,path", CASES)
def test_per_row_losses_and_gradients_match_oracle(pkg, N, M, D, precision, variant, hybrid, path):
    from speaker_embedding_ge2e_loss_b200 import _lib
    E_np = orc.make_embeddings(N, M, D, seed=N + M + D, kind="clustered")
    E = torch.tensor(E_np, device=DEV)
    crit = crit_for(pkg, precision, variant, "none")
    assert crit.path_for(N, M, D) == path
    tol = TF32_TOL if path in (1, 3) else FP32_TOL
    h = pkg.lib()
    v = _lib.VARIANTS[variant]
    pcode = _lib.resolve_precision(precision, N, N, M, D, v)
    ws_plain = h.ge2e_b200_workspace_bytes(N, N, M, D, v, pcode)
    with hybrid_mode(pkg, hybrid):
        if hybrid:    # the operand copies live in the workspace: proof that the hybrid kernels are selected
            assert h.ge2e_b200_workspace_bytes(N, N, M, D, v, pcode) > ws_plain
        for name, g in upstreams(N, M, seed=N * M + D).items():
            got = run_none(crit, E, g)
            ref = forward_backward_rows(E_np, W, B, EPS, variant, g=g)
            check_vs_oracle(got, ref, g, tol, name)


@pytest.mark.parametrize("N,M,D,precision,variant", [
    (4, 8, 64, "fp32", "softmax"), (64, 10, 256, "fp32", "softmax"), (64, 10, 256, "fp32", "contrast"),
    (256, 6, 256, "fp32", "softmax"), (256, 6, 128, "tf32", "softmax"), (1024, 10, 256, "tf32", "softmax"),
])
def test_uniform_upstream_gradient_matches_sum_and_mean(pkg, N, M, D, precision, variant):
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=3 * N + D, kind="clustered"), device=DEV)
    crit_none = crit_for(pkg, precision, variant, "none")
    tol = TF32_TOL if crit_none.path_for(N, M, D) in (1, 3) else FP32_TOL
    out = {}
    for red in ("none", "sum", "mean"):
        crit = crit_none if red == "none" else crit_for(pkg, precision, variant, red)
        Eg = E.clone().requires_grad_(True)
        loss = crit(Eg)
        (loss.sum() if red == "none" else loss).backward()       # "none": an expanded (stride-0) ones upstream
        torch.cuda.synchronize()
        out[red] = (loss.detach(), Eg.grad.clone(), crit.w.grad.item(), crit.b.grad.item())
    L, dE_n, dw_n, db_n = out["none"]
    s, dE_s, dw_s, db_s = out["sum"]
    m, dE_m, dw_m, db_m = out["mean"]
    assert L.shape == (N, M) and s.dim() == 0 and m.dim() == 0
    assert abs(L.double().sum().item() - s.item()) <= tol * max(1.0, abs(s.item()))
    assert trel(dE_n, dE_s) <= tol
    assert abs(dw_n - dw_s) <= tol * max(1.0, abs(dw_s)) and abs(db_n - db_s) <= 1e-5 * N * M
    U = N * M
    assert abs(m.item() - s.item() / U) <= 1e-6 * abs(s.item() / U)
    assert trel(dE_m, dE_s / U) <= 1e-6
    assert abs(dw_m - dw_s / U) <= 1e-6 * max(1e-6, abs(dw_s / U)) and abs(db_m - db_s / U) <= 1e-6 * max(1e-6, abs(db_s / U))


def shuffled(E, seed):
    """(flat rows in the embedder's order, unperm index): flat[unperm].reshape(N, M, D) == E."""
    N, M, D = E.shape
    perm = torch.randperm(N * M, generator=torch.Generator().manual_seed(seed)).to(DEV)
    idx = torch.empty_like(perm)
    idx[perm] = torch.arange(N * M, device=DEV)
    return E.reshape(N * M, D)[perm].contiguous(), idx


@pytest.mark.parametrize("N,M,D,precision", [(64, 10, 256, "fp32"), (256, 6, 256, "fp32"), (256, 6, 128, "tf32")])
@pytest.mark.parametrize("dtype,unperm", [(torch.float32, True), (torch.bfloat16, False), (torch.float16, False),
                                          (torch.bfloat16, True)], ids=["unperm", "bf16", "fp16", "bf16-unperm"])
def test_unperm_and_half_embeddings_match_gathered_fp32(pkg, N, M, D, precision, dtype, unperm):
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + 7, kind="clustered"), device=DEV).to(dtype)
    crit = crit_for(pkg, precision, "softmax", "none")
    path = crit.path_for(N, M, D)
    tol = (TF32_TOL if path in (1, 3) else FP32_TOL) + ROUND.get(dtype, 0.0)
    g = upstreams(N, M, seed=11)["zeros_negatives"]
    L_ref, dE_ref, dw_ref, db_ref = run_none(crit, E.float(), g)          # the gathered fp32 call
    if unperm:
        flat, idx = shuffled(E, seed=N)
        L, dE_flat, dw, db = run_none(crit, flat, g, unperm=idx, speakers=N)
        assert dE_flat.shape == flat.shape
        dE = dE_flat[idx].reshape(N, M, D)          # back to logical order
    else:
        L, dE, dw, db = run_none(crit, E, g)
    assert dE.dtype == dtype and L.dtype == torch.float32 and L.shape == (N, M)
    assert trel(L, L_ref) <= 1e-6
    assert trel(dE.float(), dE_ref) <= tol
    assert abs(dw - dw_ref) <= 1e-5 * max(1.0, abs(dw_ref)) and abs(db - db_ref) <= 1e-5 * max(1.0, abs(db_ref))


@pytest.mark.parametrize("unperm", [False, True])
def test_torch_compile(pkg, unperm):
    from speaker_embedding_ge2e_loss_b200 import ge2e_loss
    N, M, D = 64, 10, 256
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=5, kind="clustered"), device=DEV)
    w, b = torch.tensor(W, device=DEV), torch.tensor(B, device=DEV)
    g = torch.tensor(upstreams(N, M, seed=2)["normal"], dtype=torch.float32, device=DEV)
    if unperm:
        E, idx = shuffled(E, seed=3)

        def fn(x, w, b):
            return ge2e_loss(x, w, b, unperm=idx, speakers=N, reduction="none")
    else:
        def fn(x, w, b):
            return ge2e_loss(x, w, b, reduction="none")
    compiled = torch.compile(fn, backend="aot_eager", fullgraph=True)
    out = {}
    for name, f in (("eager", fn), ("compiled", compiled)):
        x = E.clone().requires_grad_(True)
        ww, bb = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        L = f(x, ww, bb)
        L.backward(g)
        torch.cuda.synchronize()
        out[name] = (L.detach(), x.grad.clone(), ww.grad.item(), bb.grad.item())
    (Le, dEe, dwe, dbe), (Lc, dEc, dwc, dbc) = out["eager"], out["compiled"]
    assert Lc.shape == (N, M)
    assert trel(Lc, Le) <= 1e-6 and trel(dEc, dEe) <= 1e-6
    assert abs(dwc - dwe) <= 1e-6 * max(1.0, abs(dwe)) and abs(dbc - dbe) <= 1e-6 * max(1.0, abs(dbe))
