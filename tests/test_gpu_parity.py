"""GPU parity tests (run on the B200 box with ``-m gpu``): the CUDA path, called through the
C ABI (ctypes binding -> libge2e_b200.so), against
  * the golden vectors produced by the REAL reference class (tests/golden/make_golden.py),
  * the numpy fp64 oracle on seeded inputs, and
  * size-independent properties at BASELINE.json's full sizes.

Tolerances (BASELINE.json north_star): fp32 path 1e-5 relative (loss, dE rel-L2, dw); TF32
tensor-core path 2e-3.  db is purely eps-driven and ill-conditioned in the reference's own fp32
autograd (SURVEY.md 8(a-bis) item 12): it is checked absolutely, |db - db_fp64| <= 1e-5 * U.
"""
import numpy as np
import pytest
import torch

from conftest import golden_names
from oracle import ge2e_oracle as orc

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
TF32_TOL = 2e-3
NAMES = golden_names()


@pytest.fixture(scope="module")
def pkg():
    import speaker_embedding_ge2e_loss_b200 as p
    p.lib()  # fails loudly when the CUDA library is missing
    assert torch.cuda.is_available()
    return p


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def run_cuda(pkg, E_np, w, b, variant="softmax", precision="fp32", g=None):
    dev = torch.device("cuda:0")
    crit = pkg.GE2ELoss(None, device=dev, w=w, b=b, variant=variant, precision=precision)
    E = torch.tensor(np.asarray(E_np, dtype=np.float32), device=dev, requires_grad=True)
    loss = crit(E)
    if g is None:
        loss.backward()
    else:
        (loss * g).backward()
    torch.cuda.synchronize()
    return dict(loss=loss.item(), dE=E.grad.double().cpu().numpy(), dw=crit.w.grad.item(),
                db=crit.b.grad.item())


def check(got, ref, U, tol, dE_tol=None):
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), (got["loss"], ref["loss"])
    assert rel(got["dE"], ref["dE"]) <= (dE_tol or tol), rel(got["dE"], ref["dE"])
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"])), (got["dw"], ref["dw"])
    assert abs(got["db"] - ref["db"]) <= 1e-5 * U, (got["db"], ref["db"])


# ------------------------------------------------------------------ golden vectors (real reference)
@pytest.mark.parametrize("name", NAMES)
def test_softmax_matches_reference_golden(pkg, golden, name):
    c = golden[name]
    got = run_cuda(pkg, c.E, c.w, c.b)
    U = c.E.shape[0] * c.E.shape[1]
    # N == 1 is purely eps-driven: loss ~ 1e-6 per row and dE ~ 1e-6 too, where fp32 exp/log
    # rounding of S itself gives ~1e-4 relative on dE even in the reference (test_oracle.py).
    dE_tol = 2e-4 if name.startswith("onespk") else FP32_TOL
    check(got, c.r64, U, FP32_TOL, dE_tol)
    # and it is at least as close to fp64 truth as 4x the reference's own fp32 run
    ref_err = rel(c.r32["dE"], c.r64["dE"])
    assert rel(got["dE"], c.r64["dE"]) <= max(4 * ref_err, FP32_TOL)


@pytest.mark.parametrize("name", NAMES)
def test_contrast_matches_golden(pkg, golden, name):
    c = golden[name]
    got = run_cuda(pkg, c.E, c.w, c.b, variant="contrast")
    ref = c.rc
    assert abs(got["loss"] - ref["loss"]) <= FP32_TOL * max(1.0, abs(ref["loss"]))
    assert rel(got["dE"], ref["dE"]) <= FP32_TOL
    assert abs(got["dw"] - ref["dw"]) <= FP32_TOL * max(1.0, abs(ref["dw"]))
    assert abs(got["db"] - ref["db"]) <= FP32_TOL * max(1.0, abs(ref["db"]))


# ------------------------------------------------------------------ seeded inputs vs the oracle
CASES = [
    (4, 8, 256, "random"), (64, 10, 256, "random"), (64, 10, 256, "clustered"),
    (2, 16, 256, "raw"), (33, 3, 48, "clustered"), (256, 10, 256, "random"),
    (97, 7, 130, "raw"), (5, 2, 1024, "random"), (300, 4, 64, "clustered"),
    # utterances per speaker beyond the register-resident kernels (M > 16: streaming warp kernels;
    # M > 32: the generic shared-memory finalize), and D = 128 / 512 on the warp-per-speaker kernels
    (24, 20, 256, "clustered"), (12, 40, 128, "random"), (16, 13, 512, "raw"), (40, 5, 128, "clustered"),
]


@pytest.mark.parametrize("N,M,D,kind", CASES)
@pytest.mark.parametrize("variant", ["softmax", "contrast"])
def test_matches_oracle_seeded(pkg, N, M, D, kind, variant):
    E = orc.make_embeddings(N, M, D, seed=N + M + D, kind=kind)
    ref = orc.forward_backward(E, 10.0, -5.0, 1e-6, variant)
    got = run_cuda(pkg, E, 10.0, -5.0, variant=variant)
    check(got, ref, N * M, FP32_TOL)


def test_upstream_gradient_scales(pkg):
    E = orc.make_embeddings(16, 5, 64, seed=5, kind="clustered")
    for variant in ("softmax", "contrast"):
        ref = orc.forward_backward(E, 3.0, -1.0, 1e-6, variant, g=-0.37)
        got = run_cuda(pkg, E, 3.0, -1.0, variant=variant, g=-0.37)
        check(got, ref, 80, FP32_TOL)


def test_forward_only_and_repeat_is_deterministic_loss(pkg):
    # s4:103: the test-loss path calls forward with grad enabled and never backpropagates
    dev = torch.device("cuda:0")
    crit = pkg.GE2ELoss(None, device=dev)
    E = torch.tensor(orc.make_embeddings(32, 6, 256, seed=9), device=dev, requires_grad=True)
    l1 = crit(E)
    l2 = crit(E)
    with torch.no_grad():
        l3 = crit(E)
    torch.cuda.synchronize()
    assert abs(l1.item() - l2.item()) <= 1e-6 * abs(l1.item())
    assert abs(l1.item() - l3.item()) <= 1e-6 * abs(l1.item())
    assert not l3.requires_grad and l1.requires_grad


# ------------------------------------------------------------------ full-size properties
@pytest.mark.parametrize("precision,tol", [("fp32", FP32_TOL), ("tf32", TF32_TOL)])
def test_cfg3_full_size_vs_oracle(pkg, precision, tol):
    # N=1024, M=10, D=256: the reference cannot run this (>80 GB); the fp64 oracle can.
    N, M, D = 1024, 10, 256
    E = orc.make_embeddings(N, M, D, seed=3, kind="clustered")
    ref = orc.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
    got = run_cuda(pkg, E, 10.0, -5.0, precision=precision)
    check(got, ref, N * M, tol)


@pytest.mark.parametrize("precision,tol", [("fp32", FP32_TOL), ("tf32", TF32_TOL)])
def test_cfg3_contrast_vs_oracle(pkg, precision, tol):
    N, M, D = 1024, 10, 256
    E = orc.make_embeddings(N, M, D, seed=4, kind="random")
    ref = orc.forward_backward(E, 10.0, -5.0, 1e-6, "contrast")
    got = run_cuda(pkg, E, 10.0, -5.0, variant="contrast", precision=precision)
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"]))
    if precision == "fp32":
        assert rel(got["dE"], ref["dE"]) <= tol
    else:
        # TF32 rounding may move the argmax between near-tied negatives; compare what is robust
        assert abs(got["dw"] - ref["dw"]) <= 5e-2 * max(1.0, abs(ref["dw"]))


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_large_n_properties(pkg, precision):
    """N=8192, M=16, D=256 (cfg 4) on one GPU: properties that do not need the O(U N D) oracle.
      * sum_k p_rk < 1 => per-row loss >= 0 and loss is finite;
      * permuting speakers permutes dE and leaves loss, dw, db unchanged (up to summation order);
      * a row sample of per-row losses equals the oracle evaluated on those rows only."""
    tol = FP32_TOL if precision == "fp32" else TF32_TOL
    N, M, D = 8192, 16, 256
    dev = torch.device("cuda:0")
    E_np = orc.make_embeddings(N, M, D, seed=11, kind="clustered")
    got = run_cuda(pkg, E_np, 10.0, -5.0, precision=precision)
    assert np.isfinite(got["loss"]) and np.isfinite(got["dE"]).all()
    perm = np.random.default_rng(0).permutation(N)
    got_p = run_cuda(pkg, E_np[perm], 10.0, -5.0, precision=precision)
    assert abs(got_p["loss"] - got["loss"]) <= tol * abs(got["loss"])
    assert abs(got_p["dw"] - got["dw"]) <= tol * max(1.0, abs(got["dw"]))
    assert rel(got_p["dE"], got["dE"][perm]) <= tol
    # row sample against the oracle's definition (rows of 3 speakers against all centroids)
    E64 = E_np.astype(np.float64)
    C = E64.mean(axis=1)
    Ch = C / np.maximum(np.linalg.norm(C, axis=1, keepdims=True), 1e-8)
    spk = [0, 4097, 8191]
    want = 0.0
    for j in spk:
        e = E64[j]
        eh = e / np.maximum(np.linalg.norm(e, axis=1, keepdims=True), 1e-8)
        u = (e.sum(0, keepdims=True) - e) / (M - 1)
        uh = u / np.maximum(np.linalg.norm(u, axis=1, keepdims=True), 1e-8)
        cos = eh @ Ch.T
        cos[:, j] = (eh * uh).sum(1)
        S = 10.0 * (cos + 1e-6) - 5.0
        want += (np.log(np.exp(S).sum(1) + 1e-6) - S[:, j]).sum()
    crit = pkg.GE2ELoss(None, device=dev)
    Et = torch.tensor(E_np, device=dev)
    sim = pkg.GE2ELoss.get_cos_sim(Et, None)            # fp32 path, materialised [N, M, N]
    _, per = pkg.GE2ELoss.calc_loss(crit.w.detach() * sim + crit.b.detach())
    have = per[spk].double().sum().item()
    assert abs(have - want) <= FP32_TOL * abs(want)
    assert abs(per.double().sum().item() - got["loss"]) <= tol * abs(got["loss"])


# ------------------------------------------------------------------ tensor-core path: shapes and schedules
# (N, M, D, kind): row tails (N*M and N not multiples of 128), every D the TMA slabs allow, M = 2,
# the "whole dE groups + dC filler" schedule (1024x10, 700x9) and the flat fallback cut (2048x2: few
# utterance tiles against many centroids)
TC_CASES = [
    (300, 7, 64, "clustered"), (300, 7, 96, "random"), (257, 5, 128, "clustered"), (700, 9, 256, "random"),
    (2048, 2, 256, "clustered"), (513, 3, 32, "random"), (1024, 10, 256, "random"),
    (256, 20, 256, "clustered"), (260, 40, 128, "random"),
]


@pytest.mark.parametrize("N,M,D,kind", TC_CASES)
def test_tensor_core_path_vs_oracle(pkg, N, M, D, kind):
    assert pkg.lib().ge2e_b200_path(N, N, M, D, 0, 1) == 1, "shape should take the tcgen05 path"
    E = orc.make_embeddings(N, M, D, seed=N + 3 * M + D, kind=kind)
    ref = orc.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
    got = run_cuda(pkg, E, 10.0, -5.0, precision="tf32")
    check(got, ref, N * M, TF32_TOL)
    # the fp32 SIMT path on the same batch pins the tensor-core path much tighter than 2e-3 in practice
    exact = run_cuda(pkg, E, 10.0, -5.0, precision="fp32")
    assert rel(got["dE"], exact["dE"]) <= 5e-4
    assert abs(got["loss"] - exact["loss"]) <= 1e-5 * abs(exact["loss"])


def test_tensor_core_negative_w_and_upstream_gradient(pkg):
    # w is not clamped (s3:22 is a no-op): negative w is legal; upstream gradient g != 1
    N, M, D = 384, 4, 128
    E = orc.make_embeddings(N, M, D, seed=21, kind="clustered")
    ref = orc.forward_backward(E, -3.0, 0.5, 1e-6, "softmax", g=0.25)
    got = run_cuda(pkg, E, -3.0, 0.5, precision="tf32", g=0.25)
    check(got, ref, N * M, TF32_TOL)


def test_tensor_core_repeated_backward_and_reuse(pkg):
    """The workspace is zero on entry and must be zero again on exit (stream-K bookkeeping, grid
    counters): a second backward through the same graph and a second forward+backward on the same
    module must reproduce the first results."""
    dev = torch.device("cuda:0")
    N, M, D = 640, 6, 256
    E_np = orc.make_embeddings(N, M, D, seed=5, kind="clustered")
    crit = pkg.GE2ELoss(None, device=dev, precision="tf32")
    E = torch.tensor(E_np, device=dev, requires_grad=True)
    loss = crit(E)
    loss.backward(retain_graph=True)
    g1 = E.grad.clone()
    E.grad = None
    loss.backward()
    torch.cuda.synchronize()
    assert rel(E.grad.cpu().numpy(), g1.cpu().numpy()) <= 5e-6
    plan = pkg.GE2EPlan(N, M, D, "softmax", "tf32", device=dev)
    w = torch.tensor(10.0, device=dev)
    b = torch.tensor(-5.0, device=dev)
    Ed = torch.tensor(E_np, device=dev)
    outs = []
    for _ in range(3):                    # same persistent workspace three times
        plan.step(Ed, w, b)
        torch.cuda.synchronize()
        outs.append((plan.loss.item(), plan.dE.clone(), plan.dw.item()))
    for o in outs[1:]:
        assert abs(o[0] - outs[0][0]) <= 1e-6 * abs(outs[0][0])
        assert rel(o[1].cpu().numpy(), outs[0][1].cpu().numpy()) <= 5e-6
    assert rel(outs[0][1].cpu().numpy().reshape(-1), g1.cpu().numpy().reshape(-1)) <= 5e-6


def test_custom_op_path_matches_eager_path(pkg):
    """The torch.library ops (what torch.compile / export trace) and the lean eager autograd.Function
    drive the same C-ABI calls: same loss and gradients, on both kernel paths."""
    from speaker_embedding_ge2e_loss_b200 import ops
    dev = torch.device("cuda:0")
    for (N, M, D, prec) in ((48, 5, 128, "fp32"), (320, 4, 256, "tf32")):
        E_np = orc.make_embeddings(N, M, D, seed=N, kind="clustered")
        res = []
        for use_op in (False, True):
            E = torch.tensor(E_np, device=dev, requires_grad=True)
            w = torch.tensor(10.0, device=dev, requires_grad=True)
            b = torch.tensor(-5.0, device=dev, requires_grad=True)
            if use_op:
                loss = torch.ops.ge2e_b200.fwd(E, w, b, 1e-6, 0, 0 if prec == "fp32" else 1)[0]
            else:
                loss = ops.ge2e_loss(E, w, b, 1e-6, "softmax", prec)
            loss.backward()
            torch.cuda.synchronize()
            res.append((loss.item(), E.grad.cpu().numpy(), w.grad.item(), b.grad.item()))
        assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[0][0])
        assert rel(res[1][1], res[0][1]) <= 5e-6
        assert abs(res[0][2] - res[1][2]) <= 1e-5 * max(1.0, abs(res[0][2]))


@pytest.mark.parametrize("N,M,D,precision", [(6, 5, 64, "fp32"), (64, 10, 256, "fp32"), (320, 6, 256, "tf32"),
                                             (40, 20, 128, "fp32"), (24, 40, 96, "fp32")])
def test_unperm_fused_matches_gather(pkg, N, M, D, precision):
    """SURVEY 8(f) row 1: ``crit(flat, unperm=idx, speakers=N)`` == ``crit(flat[idx].reshape(N, M, D))``
    (s4_train_embed_model.py:177-192), including the gradient scattered back to flat's row order."""
    dev = torch.device("cuda:0")
    E_np = orc.make_embeddings(N, M, D, seed=N * M, kind="clustered").reshape(N * M, D)
    rng = np.random.default_rng(1)
    perm = rng.permutation(N * M)
    unperm = np.argsort(perm)
    flat_np = E_np[perm]                      # the embedder saw the rows in shuffled order
    assert np.array_equal(flat_np[unperm], E_np)
    idx = torch.tensor(unperm, device=dev)
    res = []
    for fused in (False, True):
        crit = pkg.GE2ELoss(None, device=dev, precision=precision)
        flat = torch.tensor(flat_np, device=dev, requires_grad=True)
        loss = crit(flat, unperm=idx, speakers=N) if fused else crit(flat[idx].reshape(N, M, D))
        loss.backward()
        torch.cuda.synchronize()
        res.append((loss.item(), flat.grad.cpu().numpy(), crit.w.grad.item()))
    assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[0][0])
    assert rel(res[1][1], res[0][1]) <= 5e-6
    assert abs(res[0][2] - res[1][2]) <= 1e-5 * max(1.0, abs(res[0][2]))
    ref = orc.forward_backward(E_np.reshape(N, M, D), 10.0, -5.0, 1e-6, "softmax")
    tol = FP32_TOL if precision == "fp32" else TF32_TOL
    assert abs(res[1][0] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"]))
    assert rel(res[1][1][unperm], ref["dE"].reshape(N * M, D)) <= tol


# ------------------------------------------------------------------ static helpers (s5:42-43)
def test_static_helpers_match_oracle(pkg):
    dev = torch.device("cuda:0")
    E_np = orc.make_embeddings(12, 5, 100, seed=2, kind="raw")
    E = torch.tensor(E_np, device=dev)
    C = pkg.GE2ELoss.get_centroids(E)
    np.testing.assert_allclose(C.cpu().numpy(), orc.get_centroids(E_np), rtol=1e-5, atol=1e-6)
    Uc = pkg.GE2ELoss.get_utterance_centroids(E)
    np.testing.assert_allclose(Uc.cpu().numpy(), orc.get_utterance_centroids(E_np), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(pkg.GE2ELoss.get_centroid(E, 3, 2).cpu().numpy(),
                               orc.get_utterance_centroids(E_np)[3, 2], rtol=1e-5, atol=1e-6)
    cos = pkg.GE2ELoss.get_cos_sim(E, C)
    np.testing.assert_allclose(cos.cpu().numpy(), orc.get_cos_sim(E_np, 1e-6), rtol=0, atol=2e-6)
    S = 10.0 * cos - 5.0
    loss, per = pkg.GE2ELoss.calc_loss(S)
    want, want_per = orc.calc_loss(S.double().cpu().numpy(), 1e-6)
    assert abs(loss.item() - want) <= FP32_TOL * abs(want)
    np.testing.assert_allclose(per.cpu().numpy(), want_per, rtol=1e-5, atol=1e-5)
    loss_c, per_c = pkg.GE2ELoss.calc_loss(S, variant="contrast")
    want_c, want_per_c, _ = orc.calc_loss_contrast(S.double().cpu().numpy())
    assert abs(loss_c.item() - want_c) <= FP32_TOL * abs(want_c)


def test_eval_call_pattern_s5(pkg):
    # s5_eval_model.py:27-28,42-46: CPU 0-dim w=1, b=0 and sim = w*cos+b then .numpy()
    dev = torch.device("cuda:0")
    E_np = orc.make_embeddings(4, 8, 256, seed=1)
    E = torch.tensor(E_np, device=dev)
    cent = pkg.GE2ELoss.get_centroids(E)
    cos = pkg.GE2ELoss.get_cos_sim(E, cent, None)
    sim = (1.0 * cos + 0.0).detach().cpu().numpy()
    np.testing.assert_allclose(sim, orc.get_cos_sim(E_np, 1e-6), atol=2e-6)


# ------------------------------------------------------------------ error behaviour
def test_errors(pkg):
    dev = torch.device("cuda:0")
    crit = pkg.GE2ELoss(None, device=dev)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.ge2e_loss(torch.zeros(2, 3, 4), torch.tensor(10.0), torch.tensor(-5.0))
    with pytest.raises(ValueError):
        crit(torch.zeros(2, 1, 4, device=dev))          # M == 1: reference yields NaN (s3:110-111)
    with pytest.raises(ValueError):
        crit(torch.zeros(6, 4, device=dev))
    with pytest.raises(TypeError):
        crit(torch.zeros(2, 3, 4, device=dev, dtype=torch.float64))
    with pytest.raises(ValueError):
        pkg.GE2ELoss(None, device=dev, variant="triplet")
    # all-zero embeddings are finite (cos = 0)
    E = torch.zeros(3, 4, 32, device=dev, requires_grad=True)
    loss = crit(E)
    loss.backward()
    assert torch.isfinite(loss) and torch.isfinite(E.grad).all()
    # non-contiguous input is accepted (made contiguous), as the reference's .view would require
    Ebig = torch.tensor(orc.make_embeddings(4, 6, 64, seed=3), device=dev)
    Enc = Ebig.transpose(0, 1).contiguous().transpose(0, 1)
    assert abs(crit(Enc).item() - crit(Ebig).item()) < 1e-5


# ------------------------------------------------------------------ drop-in training loop (s4:188-205)
def test_training_steps_track_reference_port(pkg):
    """The s4 step sequence (two SGD param groups, clip 3.0 / 1.0, loss.to('cpu')) with the CUDA
    loss vs the torch port of the reference's expanded algorithm on CPU: same trajectories."""
    from oracle import ge2e_ref_port as port
    dev = torch.device("cuda:0")
    N, M, F, D = 8, 6, 24, 64
    torch.manual_seed(0)
    X = torch.randn(N * M, F)
    spk = torch.randn(N, 1, F).repeat(1, M, 1).reshape(N * M, F)
    X = X * 0.3 + spk

    def make(device):
        torch.manual_seed(1)
        lin = torch.nn.Linear(F, D)
        return lin.to(device)

    class RefLoss(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.tensor(10.0))
            self.b = torch.nn.Parameter(torch.tensor(-5.0))

        def forward(self, E):
            return port.loss_full(E, self.w, self.b, 1e-6)

    traj = {}
    for tag, device, crit in (("ref", torch.device("cpu"), RefLoss()),
                              ("new", dev, pkg.GE2ELoss(None, device=dev))):
        model = make(device)
        opt = torch.optim.SGD([{"params": model.parameters()}, {"params": crit.parameters()}], lr=0.01)
        losses = []
        x = X.to(device)
        for _ in range(8):
            emb = model(x)
            emb = emb / emb.norm(dim=1, keepdim=True)          # s2:34
            loss = crit(emb.reshape(N, M, D))                   # s4:192-196
            opt.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 3.0)
            torch.nn.utils.clip_grad_norm_(crit.parameters(), 1.0)
            opt.step()
            losses.append(float(loss.to("cpu").detach().numpy()))
        traj[tag] = (losses, crit.w.item(), crit.b.item())
    np.testing.assert_allclose(traj["new"][0], traj["ref"][0], rtol=2e-4)
    assert abs(traj["new"][1] - traj["ref"][1]) < 1e-4
    assert abs(traj["new"][2] - traj["ref"][2]) < 1e-4


@pytest.mark.parametrize("N,M,D,precision,tol", [(96, 6, 256, "tf32", 2e-3), (40, 5, 128, "fp32", 1e-5)])
def test_host_feed_matches_oracle_per_batch(pkg, N, M, D, precision, tol):
    """GE2EHostFeed (bench.py's e2e arm): pinned host batches in, {loss, dw, db} read back per step,
    copy of batch k+1 under the step of batch k.  Every batch's result must be that batch's oracle
    result, in order, with more batches than slots (slot reuse) and an in-place update of w between
    submits (w is read at replay time)."""
    dev = torch.device("cuda:0")
    w = torch.tensor(10.0, device=dev)
    b = torch.tensor(-5.0, device=dev)
    feed = pkg.GE2EHostFeed(N, M, D, w, b, "softmax", precision, device=dev)
    batches = [orc.make_embeddings(N, M, D, seed=s, kind="clustered") for s in range(5)]
    hosts = [torch.tensor(np.asarray(x, dtype=np.float32)).pin_memory() for x in batches]
    tickets, got, dEs = [], [], []
    for k, h in enumerate(hosts):
        if k == 3:
            torch.cuda.synchronize()
            w.fill_(7.5)
        t = feed.submit(h)
        if tickets:
            got.append(feed.result(tickets[-1]))
        tickets.append(t)
        feed.done_event(t).synchronize()
        dEs.append(feed.dE(t).cpu().numpy().copy())
    got.append(feed.result(tickets[-1]))
    for k, x in enumerate(batches):
        ref = orc.forward_backward(x, 10.0 if k < 3 else 7.5, -5.0, 1e-6, "softmax")
        check(dict(loss=got[k][0], dw=got[k][1], db=got[k][2], dE=dEs[k]), ref, N * M, tol)
    with pytest.raises(ValueError):
        feed.submit(torch.zeros(N, M, D))            # unpinned host memory


def test_clip_and_sgd_tail_matches_torch(pkg):
    """SURVEY 8(f) row 1, second half: clip_grad_norm_((w, b), 1.0) + SGD step of the loss parameters
    (s4:202-203) as one kernel, against torch's own two calls on the same gradients -- with the norm
    above max_norm (the usual case at training sizes) and below it."""
    dev = torch.device("cuda:0")
    N, M, D = 16, 5, 64
    E_np = orc.make_embeddings(N, M, D, seed=2, kind="clustered")
    for scale, lr in ((100.0, 0.01), (1.0, 0.5)):
        ours = pkg.GE2ELoss(None, device=dev)
        E = torch.tensor(np.asarray(E_np, dtype=np.float32), device=dev)
        (ours(E) * scale).backward()
        ref_w = torch.nn.Parameter(ours.w.detach().clone())
        ref_b = torch.nn.Parameter(ours.b.detach().clone())
        ref_w.grad, ref_b.grad = ours.w.grad.clone(), ours.b.grad.clone()
        ref_norm = torch.nn.utils.clip_grad_norm_([ref_w, ref_b], 1.0)
        torch.optim.SGD([ref_w, ref_b], lr=lr).step()
        norm = ours.clip_and_sgd_step(lr=lr, max_norm=1.0, return_norm=True)
        torch.cuda.synchronize()
        assert (ref_norm.item() > 1.0) == (scale == 100.0)
        for got, ref in ((norm, ref_norm), (ours.w, ref_w), (ours.b, ref_b), (ours.w.grad, ref_w.grad),
                         (ours.b.grad, ref_b.grad)):
            assert abs(got.item() - ref.item()) <= 2e-6 * max(1.0, abs(ref.item())), (got.item(), ref.item())
    with pytest.raises(RuntimeError):
        pkg.GE2ELoss(None, device=dev).clip_and_sgd_step(lr=0.01)


def test_plan_with_sgd_tail_tracks_manual_updates(pkg):
    """GE2EPlan(sgd=(lr, max_norm)): three captured steps, each ending with the fused tail, against the
    same three steps with the update applied by torch between plan steps."""
    dev = torch.device("cuda:0")
    N, M, D, lr = 64, 6, 256, 0.05
    Es = [torch.tensor(np.asarray(orc.make_embeddings(N, M, D, seed=s, kind="clustered"), dtype=np.float32), device=dev)
          for s in range(3)]
    w = torch.tensor(10.0, device=dev); b = torch.tensor(-5.0, device=dev)
    plan = pkg.GE2EPlan(N, M, D, "softmax", "tf32", device=dev, sgd=(lr, 1.0))
    g = plan.capture(Es, w, b, steps=3)
    w.fill_(10.0); b.fill_(-5.0)                         # capture's warm-up step has already moved them
    g.replay()
    torch.cuda.synchronize()
    rw = torch.nn.Parameter(torch.tensor(10.0, device=dev)); rb = torch.nn.Parameter(torch.tensor(-5.0, device=dev))
    ref = pkg.GE2EPlan(N, M, D, "softmax", "tf32", device=dev)
    for k in range(3):
        ref.step(Es[k], rw.data, rb.data)
        torch.cuda.synchronize()
        rw.grad, rb.grad = ref.dw.clone(), ref.db.clone()
        torch.nn.utils.clip_grad_norm_([rw, rb], 1.0)
        torch.optim.SGD([rw, rb], lr=lr).step()
    assert abs(w.item() - rw.item()) <= 1e-5 and abs(b.item() - rb.item()) <= 1e-5, (w.item(), rw.item(), b.item(), rb.item())
    assert abs(w.item() - 10.0) > 1e-3                   # the parameters did move
    assert abs(plan.loss.item() - ref.loss.item()) <= 1e-5 * abs(ref.loss.item())


@pytest.mark.parametrize("N,precision,tol", [(512, "fp32", 1e-5), (1024, "fp32", 1e-5), (1024, "tf32", 2e-3)])
def test_full_size_vs_reference_formulation_on_the_gpu(pkg, N, precision, tol):
    """cfg3 at FULL size against the reference's own formulation (oracle/ge2e_ref_port.py: the expanded
    repeat + F.cosine_similarity algorithm of s3:19-127 under torch autograd), which does not fit host
    memory at N=1024 but does fit the B200's HBM (86 GB peak) when run on the device.  Skipped if the
    device cannot give it that much memory."""
    from oracle import ge2e_ref_port as port
    dev = torch.device("cuda:0")
    M, D = 10, 256
    E_np = orc.make_embeddings(N, M, D, seed=1, kind="random")
    try:
        E = torch.tensor(np.asarray(E_np, dtype=np.float32), device=dev, requires_grad=True)
        w = torch.tensor(10.0, device=dev, requires_grad=True)
        b = torch.tensor(-5.0, device=dev, requires_grad=True)
        loss = port.loss_full(E, w, b)
        loss.backward()
        torch.cuda.synchronize()
        ref = dict(loss=loss.item(), dE=E.grad.double().cpu().numpy(), dw=w.grad.item(), db=b.grad.item())
        del loss, E
    except torch.OutOfMemoryError:
        torch.cuda.empty_cache()
        pytest.skip("not enough free device memory for the reference's expanded formulation")
    torch.cuda.empty_cache()
    got = run_cuda(pkg, E_np, 10.0, -5.0, precision=precision)
    assert abs(got["loss"] - ref["loss"]) <= tol * abs(ref["loss"])
    assert rel(got["dE"], ref["dE"]) <= tol
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"]))
    # db is epsilon-driven and cancels catastrophically in the reference's own fp32 autograd (SURVEY 8a-bis
    # item 12): bounded, not matched
    assert abs(got["db"] - ref["db"]) <= 1e-5 * N * M


SMALL_SHAPES = [(4, 8, 256), (64, 10, 256), (3, 2, 64), (1, 5, 32), (128, 16, 256), (7, 3, 100), (16, 6, 30), (5, 4, 7),
                (100, 10, 128),
                # fast path (D % 64 == 0) with odd M, every cluster size up to 8, D = 192, N just past the cluster limit
                (6, 16, 192), (2, 3, 128), (8, 13, 256), (9, 5, 64), (33, 7, 64), (1, 2, 256)]


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("N,M,D", SMALL_SHAPES)
def test_single_kernel_step_matches_oracle(pkg, N, M, D, variant):
    """Reference-sized batches run fwd+bwd as ONE kernel through GE2EPlan / ge2e_b200_forward_backward
    (one CTA per speaker, grid-wide barriers).  fp32 parity bar (1e-5) against the fp64 oracle, three
    steps on the same persistent workspace (its header must come back to zero), then an upstream
    gradient != 1 and a negative w."""
    dev = torch.device("cuda:0")
    pkg.lib().ge2e_b200_debug_small_step(2)                    # every supported shape, not only N <= 64
    try:
        plan = pkg.GE2EPlan(N, M, D, variant, "fp32", device=dev)
    finally:
        pkg.lib().ge2e_b200_debug_small_step(1)
    assert plan.single_kernel
    pkg.lib().ge2e_b200_debug_small_step(2)
    E_np = orc.make_embeddings(N, M, D, seed=N * 7 + M, kind="clustered")
    E = torch.tensor(np.asarray(E_np, dtype=np.float32), device=dev)
    for (wv, bv, gv) in ((10.0, -5.0, 1.0), (10.0, -5.0, 1.0), (-3.0, 0.5, 0.25)):
        w = torch.tensor(wv, device=dev)
        b = torch.tensor(bv, device=dev)
        plan.grad_out.fill_(gv)
        plan.step(E, w, b)
        torch.cuda.synchronize()
        ref = orc.forward_backward(E_np, wv, bv, 1e-6, variant, g=gv)
        got = dict(loss=plan.loss.item(), dE=plan.dE.double().cpu().numpy(), dw=plan.dw.item(), db=plan.db.item())
        check(got, ref, N * M, 1e-5)
    pkg.lib().ge2e_b200_debug_small_step(1)
    assert int(plan._ws[:256].max()) == 0                      # barrier counters restored
    default_plan = pkg.GE2EPlan(N, M, D, variant, "fp32", device=dev)
    assert default_plan.single_kernel                          # measured faster than the pipeline up to N = 128


def test_single_kernel_step_in_a_graph_and_vs_pipeline(pkg):
    """The same step captured in a CUDA graph (4 steps over 2 batches) equals the eager module API, which
    takes the multi-kernel pipeline; and the launch count of the plan is one kernel per step."""
    dev = torch.device("cuda:0")
    N, M, D = 64, 10, 256
    Es = [torch.tensor(np.asarray(orc.make_embeddings(N, M, D, seed=s, kind="clustered"), dtype=np.float32), device=dev)
          for s in (1, 2)]
    w = torch.tensor(10.0, device=dev); b = torch.tensor(-5.0, device=dev)
    pkg.lib().ge2e_b200_debug_small_step(2)
    try:
        plan = pkg.GE2EPlan(N, M, D, "softmax", "fp32", device=dev)
        g = plan.capture(Es, w, b, steps=4)
    finally:
        pkg.lib().ge2e_b200_debug_small_step(1)
    assert plan.launches_per_step == 1
    g.replay(); g.replay()
    torch.cuda.synchronize()
    ref = run_cuda(pkg, Es[1].cpu().numpy(), 10.0, -5.0)       # last step of the graph ran on Es[1]
    assert abs(plan.loss.item() - ref["loss"]) <= 1e-6 * abs(ref["loss"])
    assert rel(plan.dE.double().cpu().numpy(), ref["dE"]) <= 2e-6
    assert abs(plan.dw.item() - ref["dw"]) <= 1e-5 * max(1.0, abs(ref["dw"]))


def test_single_kernel_step_indexed_rows(pkg):
    """row_index (the trainer's unperm) through the single-kernel step: C ABI called directly."""
    import ctypes as C
    dev = torch.device("cuda:0")
    N, M, D = 12, 5, 64
    h = pkg.lib()
    E_np = np.asarray(orc.make_embeddings(N, M, D, seed=9, kind="clustered"), dtype=np.float32)
    perm = np.random.default_rng(0).permutation(N * M)
    idx = torch.tensor(perm.astype(np.int32), device=dev)      # logical row r lives at physical row perm[r]
    flat = torch.empty((N * M, D), device=dev)
    flat[idx.long()] = torch.tensor(E_np.reshape(N * M, D), device=dev)
    f32 = dict(dtype=torch.float32, device=dev)
    U = N * M
    e_hat, c_hat, cos_diag = torch.empty(U, D, **f32), torch.empty(N, D, **f32), torch.empty(U, **f32)
    row_stat, row_aux, kstar = torch.empty(U, **f32), torch.empty(U, **f32), torch.empty(U, dtype=torch.int32, device=dev)
    accum, dE_hat, scratch, dE = torch.empty(4, **f32), torch.empty(U, D, **f32), torch.empty(N * D, **f32), torch.empty(U, D, **f32)
    row_scale = torch.empty(U, **f32)
    w = torch.tensor(10.0, device=dev); b = torch.tensor(-5.0, device=dev); gone = torch.ones((), **f32)
    nb = h.ge2e_b200_step_workspace_bytes(N, M, D, 0, 0)
    assert nb > 0 and h.ge2e_b200_step_launches(N, M, D, 0, 0) == 1
    ws = torch.zeros(nb, dtype=torch.uint8, device=dev)
    rc = h.ge2e_b200_forward_backward(flat.data_ptr(), idx.data_ptr(), N, M, D, w.data_ptr(), b.data_ptr(), 1e-6, 0, 0,
                                      gone.data_ptr(), e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(),
                                      row_stat.data_ptr(), kstar.data_ptr(), row_aux.data_ptr(), row_scale.data_ptr(),
                                      accum.data_ptr(), dE_hat.data_ptr(), scratch.data_ptr(),
                                      dE.data_ptr(), ws.data_ptr(), nb, torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    ref = orc.forward_backward(E_np, 10.0, -5.0, 1e-6, "softmax")
    got = dict(loss=accum[0].item(), dE=dE[idx.long()].double().cpu().numpy().reshape(N, M, D), dw=accum[1].item(),
               db=accum[2].item())
    check(got, ref, U, 1e-5)
    # too small a workspace is refused, not overrun
    assert h.ge2e_b200_forward_backward(flat.data_ptr(), idx.data_ptr(), N, M, D, w.data_ptr(), b.data_ptr(), 1e-6, 0, 0,
                                        gone.data_ptr(), e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(),
                                        row_stat.data_ptr(), kstar.data_ptr(), row_aux.data_ptr(), row_scale.data_ptr(),
                                        accum.data_ptr(), dE_hat.data_ptr(), scratch.data_ptr(),
                                        dE.data_ptr(), ws.data_ptr(), 128, torch.cuda.current_stream().cuda_stream) == -4
