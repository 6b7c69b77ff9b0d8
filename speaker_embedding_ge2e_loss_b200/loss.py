"""Drop-in ``GE2ELoss`` module (reference: embedding_model_GE2E/s3_loss_function_GE2E.py:6-127).

Same constructor (``GE2ELoss(hp)`` reading ``hp.general.device`` and ``hp.general.small_err``),
same learnable 0-dim ``w`` / ``b`` parameters (10.0 / -5.0, s3:16-17), same
``forward(embeddings[N, M, D]) -> 0-dim loss`` and the same static helpers, so
``s4_train_embed_model.py`` and ``s5_eval_model.py`` can use it unchanged.  Extensions (keyword
only): ``variant`` ("softmax" | "contrast"), ``precision`` ("fp32" | "tf32"), ``reduction`` ("sum" |
"mean" | "none") and ``process_group`` (speaker-sharded multi-GPU).  CUDA (sm_100a) only: CPU tensors raise.
"""
from __future__ import annotations

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib, ops
from .sharded import sharded_ge2e_loss


def _hp_get(hp, name, default):
    try:
        return getattr(hp.general, name)
    except Exception:
        try:
            return hp["general"][name]
        except Exception:
            return default


class GE2ELoss(nn.Module):
    def __init__(self, hp=None, *, w: float = 10.0, b: float = -5.0, variant=None,
                 precision=None, eps=None, device=None, process_group=None, reduction: str = "sum"):
        super().__init__()
        # reduction="none": per-utterance losses [N, M] (calc_loss's per_embedding_loss, s3:121), differentiable
        if reduction not in ops.REDUCTIONS:
            raise ValueError(f"reduction must be one of {ops.REDUCTIONS}, got {reduction!r}")
        if reduction == "none" and process_group is not None:
            raise ValueError('reduction="none" is not supported together with a process_group')
        # the reference's trainer constructs GE2ELoss(hp) with no keywords (s4_train_embed_model.py:33):
        # the two opt-in extensions can therefore also come from hp.general (ge2e_variant / ge2e_precision);
        # absent both, the defaults reproduce the reference (softmax, fp32 arithmetic)
        variant = variant if variant is not None else _hp_get(hp, "ge2e_variant", "softmax")
        precision = precision if precision is not None else _hp_get(hp, "ge2e_precision", "fp32")
        if variant not in _lib.VARIANTS:
            raise ValueError(f"variant must be one of {sorted(_lib.VARIANTS)}")
        if precision not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}")
        self.hp = hp
        self.device = device if device is not None else _hp_get(hp, "device", torch.device("cuda"))
        self.eps = float(eps if eps is not None else _hp_get(hp, "small_err", 1e-6))
        self.variant = variant
        self.precision = precision
        self.process_group = process_group
        self.reduction = reduction
        # s3:16-17
        self.w = nn.Parameter(torch.tensor(float(w)).to(self.device), requires_grad=True)
        self.b = nn.Parameter(torch.tensor(float(b)).to(self.device), requires_grad=True)

    def forward(self, embeddings, unperm=None, speakers: int = 0):
        """``forward(embeddings[N, M, D])`` as in the reference.  Extension: ``forward(flat[N*M, D],
        unperm=idx, speakers=N)`` computes the loss of ``flat[idx].reshape(N, M, D)`` with the gather
        (and the scatter of its backward) folded into the kernels (s4_train_embed_model.py:189-192)."""
        # s3:22 is a discarded torch.clamp: w is deliberately NOT clamped.
        if self.process_group is not None:
            if unperm is not None:
                raise ValueError("unperm is not supported together with a process_group")
            loss = sharded_ge2e_loss(embeddings, self.w, self.b, self.eps, self.variant, self.precision,
                                     self.process_group)
            if self.reduction == "mean":     # the global sum over every rank's N_local * M utterances
                loss = loss / (embeddings.shape[0] * embeddings.shape[1] * dist.get_world_size(self.process_group))
            return loss
        return ops.ge2e_loss(embeddings, self.w, self.b, self.eps, self.variant, self.precision, unperm, speakers,
                             reduction=self.reduction)

    @torch.no_grad()
    def clip_and_sgd_step(self, lr: float, max_norm: float = 1.0, return_norm: bool = False):
        """The trainer's tail for the loss's own two parameters in ONE kernel launch
        (s4_train_embed_model.py:202-203): ``clip_grad_norm_(self.parameters(), max_norm)`` followed
        by the plain-SGD update ``p -= lr * p.grad``.  ``w.grad`` / ``b.grad`` are left clipped in
        place, as ``clip_grad_norm_`` leaves them.  Keep ``w`` and ``b`` out of the optimiser's
        parameter groups when using this.  Returns the unclipped norm (0-dim tensor) on request."""
        if self.w.grad is None or self.b.grad is None:
            raise RuntimeError("clip_and_sgd_step: call backward() first (w.grad / b.grad are None)")
        ops._need_cuda(self.w)
        norm = torch.empty((), dtype=torch.float32, device=self.w.device) if return_norm else None
        with torch.cuda.device(self.w.device):
            _lib.check(_lib.lib().ge2e_b200_scale_bias_sgd(
                self.w.data_ptr(), self.b.data_ptr(), self.w.grad.data_ptr(), self.b.grad.data_ptr(),
                float(max_norm), float(lr), norm.data_ptr() if return_norm else None, ops._stream()),
                "ge2e_b200_scale_bias_sgd")
        return norm

    def path_for(self, N: int, M: int, D: int) -> int:
        """Which kernels a batch of this shape runs on: 0 = SIMT fp32, 1 = tcgen05 TF32."""
        v = _lib.VARIANTS[self.variant]
        return _lib.lib().ge2e_b200_path(N, N, M, D, v, _lib.resolve_precision(self.precision, N, N, M, D, v))

    def extra_repr(self):
        return f"variant={self.variant}, precision={self.precision}, eps={self.eps}"

    # ---- static helpers (s3:33-127); eval-only CUDA kernels, not differentiable ------------
    @staticmethod
    def _as_f32(E):
        ops._need_cuda(E)
        if E.dim() != 3:
            raise ValueError(f"embeddings must be [N, M, D], got {tuple(E.shape)}")
        return E.detach().float().contiguous()

    @staticmethod
    def get_centroids(embeddings):
        """s3:33-38."""
        E = GE2ELoss._as_f32(embeddings)
        N, M, D = E.shape
        C = torch.empty((N, D), dtype=torch.float32, device=E.device)
        with torch.cuda.device(E.device):
            _lib.check(_lib.lib().ge2e_b200_centroids(E.data_ptr(), N, M, D, C.data_ptr(), ops._stream()),
                       "ge2e_b200_centroids")
        return C

    @staticmethod
    def get_utterance_centroids(embeddings):
        """s3:95-112."""
        E = GE2ELoss._as_f32(embeddings)
        N, M, D = E.shape
        Uc = torch.empty_like(E)
        with torch.cuda.device(E.device):
            _lib.check(_lib.lib().ge2e_b200_utterance_centroids(E.data_ptr(), N, M, D, Uc.data_ptr(),
                                                                ops._stream()),
                       "ge2e_b200_utterance_centroids")
        return Uc

    @staticmethod
    def get_centroid(embeddings, speaker_num, utterance_num):
        """s3:83-93 (unused by the reference's own callers)."""
        return GE2ELoss.get_utterance_centroids(embeddings)[speaker_num, utterance_num]

    @staticmethod
    def get_cos_sim(embeddings, centroids, hp=None):
        """s3:41-80: cos[j,i,k] (+eps) with the leave-one-out diagonal; [N, M, N]."""
        E = GE2ELoss._as_f32(embeddings)
        N, M, D = E.shape
        eps = float(_hp_get(hp, "small_err", 1e-6))
        dev = E.device
        c_hat = torch.empty((N, D), dtype=torch.float32, device=dev)
        e_hat, cos_diag, accum = ops.prep(E, c_hat, _lib.FP32)
        if centroids is not None:
            C = centroids.detach().to(dev).float().contiguous()
            if C.shape != (N, D):
                raise ValueError(f"centroids must be [{N}, {D}], got {tuple(C.shape)}")
            with torch.cuda.device(dev):
                _lib.check(_lib.lib().ge2e_b200_normalize_rows(C.data_ptr(), N, D, c_hat.data_ptr(),
                                                               ops._stream()), "ge2e_b200_normalize_rows")
        one = torch.ones((), dtype=torch.float32, device=dev)
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        sim = ops.fwd_rows(e_hat, c_hat, cos_diag, N, N, 0, M, D, one, zero, eps, _lib.SOFTMAX,
                           _lib.FP32, accum, sim=True)[4]
        return sim.view(N, M, N)

    @staticmethod
    def calc_loss(sim_matrix, hp=None, variant: str = "softmax"):
        """s3:114-127: (loss, per_embedding_loss[N, M]) from a similarity matrix [N, M, N]."""
        ops._need_cuda(sim_matrix)
        S = sim_matrix.detach().float().contiguous()
        N, M, N2 = S.shape
        if N != N2:
            raise ValueError(f"sim_matrix must be [N, M, N], got {tuple(S.shape)}")
        eps = float(_hp_get(hp, "small_err", 1e-6))
        loss = torch.empty((), dtype=torch.float32, device=S.device)
        per = torch.empty((N, M), dtype=torch.float32, device=S.device)
        with torch.cuda.device(S.device):
            _lib.check(_lib.lib().ge2e_b200_calc_loss(S.data_ptr(), N, M, eps, _lib.VARIANTS[variant],
                                                      loss.data_ptr(), per.data_ptr(), ops._stream()),
                       "ge2e_b200_calc_loss")
        return loss, per
