"""Chunked float64 torch restatement of ``oracle/ge2e_oracle.forward_backward`` -- TEST INFRASTRUCTURE.

Same algorithm, same reference lines (``s3:<line>`` of
``/root/reference/embedding_model_GE2E/s3_loss_function_GE2E.py``; SURVEY.md 8(a-bis) items 1-12), written
with torch tensors so that it can be evaluated in float64 ON the GPU box at sizes the numpy oracle does
not finish in seconds (BASELINE config 4: N = 8192, M = 16 -- a [131072, 8192] fp64 similarity matrix is
8.6 GB, so the rows are processed ``chunk`` at a time and S is never held whole).  It does NOT call any
product kernel: plain ``torch.matmul`` in float64 (cuBLAS DGEMM or CPU BLAS) is the independent
computation.  Parity pinning: ``tests/test_oracle.py`` checks it against the numpy oracle -- which is
pinned against the real reference class through ``tests/golden/`` -- on CPU; ``tests/test_gpu_parity.py``
repeats that on the device at config 2 before using it at configs 3 / 4.  Softmax and contrast variants.
"""
from __future__ import annotations

import torch

COS_DELTA = 1e-8  # F.cosine_similarity default eps (s3:57, s3:70)


def _unit(x):
    n = x.norm(dim=-1, keepdim=True)
    return x / n.clamp_min(COS_DELTA), n


def _unit_bwd(dxh, xh, n):
    """F.cosine_similarity's gradient of x / max(|x|, delta): clamped value, unclamped derivative x / |x|
    (see ge2e_oracle._unit_bwd): (dxh - xh (xh . dxh) s) / max(|x|, delta), s = max(|x|, delta) / |x|, 0 at x = 0."""
    proj = (xh * dxh).sum(-1, keepdim=True)
    nc = n.clamp_min(COS_DELTA)
    s = torch.where(n > 0, nc / torch.where(n > 0, n, torch.ones_like(n)), torch.zeros_like(n))
    return (dxh - xh * (proj * s)) / nc


def forward_backward(E, w=10.0, b=-5.0, eps=1e-6, variant="softmax", g=1.0, chunk=8192):
    """E: [N, M, D] tensor (any float dtype / device); computes in float64 on E's device.
    Returns dict(loss, per[N, M], dE[N, M, D] (float64 tensor), dw, db)."""
    E = E.detach().to(torch.float64)
    N, M, D = E.shape
    U = N * M
    Ef = E.reshape(U, D)
    s = E.sum(dim=1)                                          # s3:105
    C = s / M                                                 # s3:37
    Uc = ((s[:, None, :] - E) / (M - 1)).reshape(U, D)        # s3:111
    Eh, ne = _unit(Ef)
    Ch, nc = _unit(C)
    Uh, nu = _unit(Uc)
    cos_same = (Eh * Uh).sum(-1)                              # s3:57
    dev = E.device
    spk = torch.arange(N, device=dev).repeat_interleave(M)

    per = torch.empty(U, dtype=torch.float64, device=dev)
    dEh = torch.empty((U, D), dtype=torch.float64, device=dev)
    dCh = torch.zeros((N, D), dtype=torch.float64, device=dev)
    ddiag = torch.empty(U, dtype=torch.float64, device=dev)
    dw = torch.zeros((), dtype=torch.float64, device=dev)
    db = torch.zeros((), dtype=torch.float64, device=dev)
    for r0 in range(0, U, chunk):
        r1 = min(U, r0 + chunk)
        rows = torch.arange(r1 - r0, device=dev)
        sp = spk[r0:r1]
        cos = Eh[r0:r1] @ Ch.T                                # s3:70
        cos[rows, sp] = cos_same[r0:r1]                       # s3:77-78
        cos = cos + eps                                       # s3:79
        S = w * cos + b                                       # s3:27
        if variant == "softmax":
            expS = torch.exp(S)
            Z = expS.sum(1) + eps                             # s3:120 (un-stabilised, like the reference)
            per[r0:r1] = torch.log(Z) - S[rows, sp]           # s3:121
            G = expS / Z[:, None]
            G[rows, sp] -= 1.0
        elif variant == "contrast":
            G = torch.zeros_like(S)
            sd = torch.sigmoid(S[rows, sp])
            per[r0:r1] = 1.0 - sd
            G[rows, sp] = -sd * (1.0 - sd)
            if N > 1:
                Sm = S.clone()
                Sm[rows, sp] = -float("inf")
                # lowest index among equal maxima (torch.max does not promise which one it returns)
                mx = Sm.max(dim=1, keepdim=True).values
                kst = torch.where(Sm == mx, torch.arange(N, device=dev)[None, :], N).min(dim=1).values
                sn = torch.sigmoid(S[rows, kst])
                per[r0:r1] += sn
                G[rows, kst] += sn * (1.0 - sn)
        else:
            raise ValueError(variant)
        G = G * g
        dw += (G * cos).sum()
        db += G.sum()
        dcos = w * G
        ddiag[r0:r1] = dcos[rows, sp]
        dcos[rows, sp] = 0.0
        dEh[r0:r1] = dcos @ Ch
        dCh += dcos.T @ Eh[r0:r1]
    dEh += ddiag[:, None] * Uh
    dUh = ddiag[:, None] * Eh
    dEf = _unit_bwd(dEh, Eh, ne)
    dC = _unit_bwd(dCh, Ch, nc)
    dU = _unit_bwd(dUh, Uh, nu).reshape(N, M, D)
    dE = dEf.reshape(N, M, D) + dC[:, None, :] / M + (dU.sum(dim=1, keepdim=True) - dU) / (M - 1)
    return dict(loss=per.sum().item(), per=per.reshape(N, M), dE=dE, dw=dw.item(), db=db.item())
