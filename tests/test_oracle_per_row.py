"""CPU tests: the numpy oracle with a per-utterance upstream gradient (per_row_oracle.forward_backward_rows(..., g=[N, M]))
is pinned against float64 torch autograd of per.backward(g) -- the reference port's expanded softmax formulation, and
a direct transcription of the paper's contrast loss.  Tolerances are those of test_oracle.py."""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_ref_port as port
from per_row_oracle import forward_backward_rows


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def contrast_per(S):
    """Paper eq. (7) as calc_loss_contrast states it: 1 - sigma(S_jj) + max_{k != j} sigma(S_jk)."""
    N = S.size(0)
    j = list(range(N))
    per = 1.0 - torch.sigmoid(S[j, :, j])
    if N > 1:
        mask = torch.zeros_like(S, dtype=torch.bool)
        mask[j, :, j] = True
        per = per + torch.sigmoid(S.masked_fill(mask, -float("inf"))).amax(dim=2)
    return per


def autograd_per_row(E, w, b, eps, variant, g):
    Et = torch.tensor(E, dtype=torch.float64, requires_grad=True)
    wt = torch.tensor(w, dtype=torch.float64, requires_grad=True)
    bt = torch.tensor(b, dtype=torch.float64, requires_grad=True)
    S = wt * port.cos_sim_expanded(Et, eps) + bt
    per = port.softmax_loss(S, eps)[1] if variant == orc.SOFTMAX else contrast_per(S)
    per.backward(torch.tensor(g, dtype=torch.float64))
    return per.detach().numpy(), Et.grad.numpy(), wt.grad.item(), bt.grad.item()


def upstreams(N, M, seed):
    rng = np.random.default_rng(seed)
    onehot = np.zeros((N, M))
    onehot[N // 2, M - 1] = 1.0
    mixed = rng.standard_normal((N, M))
    mixed[rng.random((N, M)) < 0.3] = 0.0
    return {"normal": rng.standard_normal((N, M)), "zeros_negatives": -np.abs(mixed), "onehot": onehot,
            "all_zero": np.zeros((N, M))}


CASES = [(4, 8, 16, "random", 10.0, -5.0), (5, 3, 12, "raw", -3.0, 0.5), (7, 4, 24, "clustered", 4.0, -1.0)]


@pytest.mark.parametrize("variant", [orc.SOFTMAX, orc.CONTRAST])
@pytest.mark.parametrize("N,M,D,kind,w,b", CASES)
def test_per_row_gradient_matches_fp64_autograd(variant, N, M, D, kind, w, b):
    E = orc.make_embeddings(N, M, D, seed=N * D, kind=kind)
    for name, g in upstreams(N, M, seed=D).items():
        r = forward_backward_rows(E, w, b, 1e-6, variant, g=g)
        per, dE, dw, db = autograd_per_row(E, w, b, 1e-6, variant, g)
        np.testing.assert_allclose(r["per"], per, rtol=1e-10, atol=1e-12)
        assert abs(r["loss"] - per.sum()) <= 1e-11 * max(1.0, abs(per.sum()))
        if name == "all_zero":
            assert not np.any(r["dE"]) and r["dw"] == 0.0 and r["db"] == 0.0
            continue
        assert rel(r["dE"], dE) < 2e-7, name
        assert abs(r["dw"] - dw) <= 1e-9 * max(1.0, abs(dw)), name
        assert abs(r["db"] - db) <= 1e-9 * N * M, name


@pytest.mark.parametrize("variant", [orc.SOFTMAX, orc.CONTRAST])
def test_uniform_per_row_gradient_is_the_scalar_one(variant):
    E = orc.make_embeddings(6, 5, 20, seed=2, kind="raw")
    for g in (1.0, -0.75):
        s = orc.forward_backward(E, 10.0, -5.0, 1e-6, variant, g=g)
        a = forward_backward_rows(E, 10.0, -5.0, 1e-6, variant, g=np.full((6, 5), g))
        assert np.array_equal(s["dE"], a["dE"]) and s["dw"] == a["dw"] and s["db"] == a["db"]


def test_per_row_gradient_is_linear_in_g():
    # sum over one-hot upstream gradients = the all-ones gradient: each row's share is its own
    E = orc.make_embeddings(3, 4, 8, seed=5, kind="random")
    total = np.zeros((3, 4, 8))
    for r in range(12):
        g = np.zeros(12)
        g[r] = 1.0
        total += forward_backward_rows(E, 10.0, -5.0, 1e-6, orc.SOFTMAX, g=g.reshape(3, 4))["dE"]
    want = orc.forward_backward(E, 10.0, -5.0, 1e-6, orc.SOFTMAX, g=1.0)["dE"]
    assert rel(total, want) < 1e-12
