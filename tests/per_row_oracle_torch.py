"""Chunked float64 truth for a per-row upstream gradient g[N, M] -- TEST INFRASTRUCTURE.

oracle/ge2e_oracle_torch.forward_backward applies its upstream gradient once per chunk of utterance rows, as
``G = G * g`` with G the [rows of the chunk, N] gradient of the logits.  Handing it a ``RowGradient`` there makes that
product take the chunk's own rows of g: torch's ``G.__mul__`` does not know the object, so Python calls
``RowGradient.__rmul__(G)``, which scales row i of G by g[r0 + i] and moves r0 on by the chunk.  So the unmodified,
pinned oracle computes dE = sum_r g_r dper_r / dE at config 4 sizes (where S is never held whole) as it does for a
scalar.  test_per_row_oracle_torch.py pins the result against tests/per_row_oracle.forward_backward_rows.
"""
import torch

from oracle import ge2e_oracle_torch as orct


class RowGradient:
    """g[N, M] consumed chunk by chunk, in the order forward_backward visits its rows."""

    def __init__(self, g):
        self.g = torch.as_tensor(g).reshape(-1, 1)
        self.r0 = 0

    def __rmul__(self, G):
        n = G.shape[0]
        out = G * self.g[self.r0:self.r0 + n].to(G)
        self.r0 += n
        return out


def forward_backward_rows(E, w=10.0, b=-5.0, eps=1e-6, variant="softmax", g=1.0, chunk=8192):
    """orct.forward_backward with g a scalar (unchanged) or an [N, M] tensor of per-utterance upstream gradients."""
    if not torch.is_tensor(g) or g.dim() == 0:
        return orct.forward_backward(E, w, b, eps, variant, g=float(g), chunk=chunk)
    N, M = E.shape[:2]
    assert g.numel() == N * M, (tuple(g.shape), N, M)
    rg = RowGradient(g.to(E.device, torch.float64))
    out = orct.forward_backward(E, w, b, eps, variant, g=rg, chunk=chunk)
    assert rg.r0 == N * M, "every row of g must have been used exactly once"
    return out
