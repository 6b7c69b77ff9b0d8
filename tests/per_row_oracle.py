"""Float64 truth for the per-utterance losses and a per-row upstream gradient g[N, M] -- TEST INFRASTRUCTURE.

oracle/ge2e_oracle.forward_backward applies its upstream gradient in exactly two forms: softmax scales the whole
gradient matrix G[U, N] of the logits (``G *= g``), contrast scales the two per-row entries it writes
(``-g * sp * (1 - sp)``, ``g * sn * (1 - sn)`` with sp, sn of shape [U]).  Both are elementwise products, so the same
unmodified function computes dE = sum_r g_r dper_r/dE when g is handed over with the shape that broadcasts over
utterance rows: a column [U, 1] against G for softmax, a vector [U] for contrast.  test_oracle_per_row.py pins the
result against float64 torch autograd of per.backward(g).
"""
import numpy as np

from oracle import ge2e_oracle as orc


def forward_backward_rows(E, w=10.0, b=-5.0, eps=1e-6, variant=orc.SOFTMAX, g=1.0):
    """orc.forward_backward with g a scalar (unchanged) or an [N, M] array of per-utterance upstream gradients."""
    if np.ndim(g) == 0:
        return orc.forward_backward(E, w, b, eps, variant, g=g)
    N, M = np.shape(E)[:2]
    g = np.asarray(g, dtype=np.float64).reshape(N * M)
    return orc.forward_backward(E, w, b, eps, variant, g=g[:, None] if variant == orc.SOFTMAX else g)
