"""CPU: the chunked float64 per-row reference (tests/per_row_oracle_torch.py) equals the numpy per-row oracle
(tests/per_row_oracle.py, itself pinned against torch autograd) for chunks that cut speakers apart, and a scalar g
keeps ge2e_oracle_torch.forward_backward's own result."""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_oracle_torch as orct
from per_row_oracle import forward_backward_rows as numpy_rows
from per_row_oracle_torch import forward_backward_rows as torch_rows


def _g(kind, N, M):
    rng = np.random.default_rng(5)
    if kind == "signed":
        return rng.standard_normal((N, M))
    if kind == "mask":
        return (rng.random((N, M)) > 0.5).astype(np.float64)
    g = rng.standard_normal((N, M))
    g[: N // 2] = 0.0                       # every row of the first half of the speakers carries no gradient
    return g


@pytest.mark.parametrize("variant", ["softmax", "contrast"])
@pytest.mark.parametrize("kind", ["signed", "mask", "zero_half"])
@pytest.mark.parametrize("chunk", [7, 16, 1000])
def test_chunked_rows_equal_numpy_rows(variant, kind, chunk):
    N, M, D = 12, 4, 16
    E = orc.make_embeddings(N, M, D, seed=3, kind="clustered")
    g = _g(kind, N, M)
    ref = numpy_rows(E, 10.0, -5.0, 1e-6, variant, g=g)
    got = torch_rows(torch.tensor(E), 10.0, -5.0, 1e-6, variant, g=torch.tensor(g), chunk=chunk)
    assert np.allclose(got["per"].numpy(), ref["per"], rtol=1e-12, atol=1e-12)
    assert np.linalg.norm(got["dE"].numpy() - ref["dE"]) <= 1e-11 * max(1e-30, np.linalg.norm(ref["dE"]))
    assert abs(got["dw"] - ref["dw"]) <= 1e-11 * max(1.0, abs(ref["dw"]))
    assert abs(got["db"] - ref["db"]) <= 1e-11 * max(1.0, abs(ref["db"]))


def test_scalar_g_is_the_plain_oracle():
    E = torch.tensor(orc.make_embeddings(8, 3, 16, seed=1, kind="clustered"))
    a = torch_rows(E, 10.0, -5.0, 1e-6, "softmax", g=-1.5, chunk=5)
    b = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax", g=-1.5, chunk=5)
    assert a["loss"] == b["loss"] and a["dw"] == b["dw"] and a["db"] == b["db"] and torch.equal(a["dE"], b["dE"])
