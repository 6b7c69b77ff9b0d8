"""CPU tests: the oracles' gradients on degenerate batches -- rows, centroids and leave-one-out centroids whose
norm is at or below the cosine clamp delta = 1e-8 -- against autograd through the reference's own expanded
F.cosine_similarity formulation (oracle/ge2e_ref_port.py), in float64.

F.cosine_similarity clamps the norm's VALUE at delta but keeps the norm's derivative x / |x|, so for
0 < |x| < delta its gradient is not dxh / delta.  The well-behaved inputs of test_oracle.py never reach this
branch; the kernels implement whatever the oracles say, so the oracles must say what torch does.
"""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_oracle_torch as orct
from oracle import ge2e_ref_port as port

DELTA = orc.COS_DELTA
W, B, EPS = 10.0, -5.0, 1e-6


def _base(N=6, M=4, D=32, seed=1):
    return orc.make_embeddings(N, M, D, seed=seed, kind="clustered").astype(np.float64)


def _dir(D, seed):
    v = np.random.default_rng(seed).standard_normal(D)
    return v / np.linalg.norm(v)


def _row_norm(s):
    E = _base()
    E[0, 0] *= s * DELTA / np.linalg.norm(E[0, 0])
    return E, [0]


def _centroid_norm(s):
    # M = 2: e_2 = -e_1 + t, so c = t / 2 with |c| = s delta
    E = _base(M=2)
    E[2, 1] = -E[2, 0] + 2.0 * s * DELTA * _dir(E.shape[-1], 7)
    return E, [2]


def _loo_norm(s):
    # M = 3: e_3 = -e_2 + t, so the leave-one-out centroid of e_1 is t / 2 with |u| = s delta
    E = _base(M=3)
    E[3, 2] = -E[3, 1] + 2.0 * s * DELTA * _dir(E.shape[-1], 8)
    return E, [3]


def _zero_row():
    E = _base()
    E[2, 1] = 0.0
    return E, [2]


def _zero_centroid_m2():
    E = _base(M=2)
    E[1, 1] = -E[1, 0]
    return E, [1]


def _zero_centroid_m4():
    E = _base(M=4)
    E[3, 1] = -E[3, 0]
    E[3, 2] = -E[3, 3]
    return E, [3]


def _zero_loo_m3():
    E = _base(M=3)
    E[1, 1] = -E[1, 2]
    return E, [1]


def _collapsed():
    E = _base()
    E[4] = E[4, 0]
    return E, [4]


def _duplicated():
    E = _base()
    E[5] = E[0]
    return E, [0, 5]


def _single_speaker():
    return _base(N=1, M=5), []


SCALES = [0.0, 0.5, 0.999, 1.001, 2.0]
CASES = {
    "zero_row": _zero_row,
    "zero_centroid_m2": _zero_centroid_m2,
    "zero_centroid_m4": _zero_centroid_m4,
    "zero_loo_centroid_m3": _zero_loo_m3,
    "collapsed_speaker": _collapsed,
    "duplicated_speaker": _duplicated,
    "single_speaker": _single_speaker,
}
for _s in SCALES:
    CASES[f"row_norm_{_s}delta"] = (lambda s: lambda: _row_norm(s))(_s)
    CASES[f"centroid_norm_{_s}delta"] = (lambda s: lambda: _centroid_norm(s))(_s)
    CASES[f"loo_norm_{_s}delta"] = (lambda s: lambda: _loo_norm(s))(_s)


def autograd_ref(E, w=W, b=B, g=1.0):
    Et = torch.tensor(E, dtype=torch.float64, requires_grad=True)
    wt = torch.tensor(w, dtype=torch.float64, requires_grad=True)
    bt = torch.tensor(b, dtype=torch.float64, requires_grad=True)
    loss = port.loss_full(Et, wt, bt, EPS)
    (loss * g).backward()
    return dict(loss=loss.item(), dE=Et.grad.numpy(), dw=wt.grad.item(), db=bt.grad.item())


def rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def check(got, ref, degenerate, tol=1e-8):
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), (got["loss"], ref["loss"])
    dE, rE = np.asarray(got["dE"]), ref["dE"]
    N = rE.shape[0]
    # the degenerate speakers' gradients can be ~1/delta: compare them and the other rows separately
    normal = [j for j in range(N) if j not in degenerate]
    if degenerate:
        assert rel(dE[degenerate], rE[degenerate]) <= tol, rel(dE[degenerate], rE[degenerate])
    if normal:
        assert rel(dE[normal], rE[normal]) <= tol, rel(dE[normal], rE[normal])
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"])), (got["dw"], ref["dw"])
    assert abs(got["db"] - ref["db"]) <= tol * max(1.0, abs(ref["db"])), (got["db"], ref["db"])


@pytest.mark.parametrize("case", sorted(CASES))
def test_numpy_oracle_matches_reference_autograd(case):
    E, degenerate = CASES[case]()
    ref = autograd_ref(E)
    got = orc.forward_backward(E, W, B, EPS, orc.SOFTMAX)
    assert np.isfinite(got["dE"]).all()
    check(got, ref, degenerate)


@pytest.mark.parametrize("case", sorted(CASES))
def test_torch_oracle_matches_reference_autograd(case):
    E, degenerate = CASES[case]()
    g = -0.7
    ref = autograd_ref(E, g=g)
    got = orct.forward_backward(torch.tensor(E), W, B, EPS, "softmax", g=g, chunk=7)
    got["dE"] = got["dE"].numpy()
    check(got, ref, degenerate)
    ref_loss = autograd_ref(E)["loss"]          # the loss is not scaled by g
    assert abs(got["loss"] - ref_loss) <= 1e-9 * max(1.0, abs(ref_loss))


@pytest.mark.parametrize("s", [0.5, 0.999])
def test_single_cosine_pair_gradient_below_the_clamp(s):
    """The formula in isolation: one F.cosine_similarity pair with |x| = s delta."""
    D = 8
    x = torch.tensor(_dir(D, 3) * s * DELTA, requires_grad=True)
    y = torch.tensor(_dir(D, 4))
    torch.nn.functional.cosine_similarity(x[None], y[None]).sum().backward()
    xh, n, _ = orc._unit(x.detach().numpy())
    yh = y.numpy() / np.linalg.norm(y.numpy())
    got = orc._unit_bwd(yh, xh, n)
    assert rel(got, x.grad.numpy()) <= 1e-12
    # the old spec (dxh / delta) is measurably different here: the test can tell the two apart
    assert rel(yh / DELTA, x.grad.numpy()) > 1e-3
