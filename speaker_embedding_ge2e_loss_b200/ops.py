"""torch.library custom ops over the C ABI (CUDA only; raises on CPU tensors).

``ge2e_b200::fwd`` / ``ge2e_b200::bwd`` are the single-device ops; the staged ops
(``prep``, ``fwd_rows``, ``bwd_rows``, ``bwd_finalize``) are what the speaker-sharded
autograd function in ``sharded.py`` strings together around its collectives.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import check, lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts: Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("speaker_embedding_ge2e_loss_b200 runs on CUDA (sm_100a) tensors only; "
                               "there is no CPU fallback")


def _f32c(t: Tensor) -> Tensor:
    if t.dtype != torch.float32:
        raise TypeError(f"expected float32, got {t.dtype}")
    return t.contiguous()


# element types the kernels read E in (and write dE in): ge2e_dtype codes of include/ge2e_b200.h
_DTYPES = {torch.float32: _lib.DT_F32, torch.bfloat16: _lib.DT_BF16, torch.float16: _lib.DT_F16}


def _emb(E: Tensor) -> Tuple[Tensor, int]:
    """E contiguous, with its ge2e_dtype code: float32, bfloat16 or float16 embeddings."""
    code = _DTYPES.get(E.dtype)
    if code is None:
        raise TypeError(f"embeddings must be float32, bfloat16 or float16, got {E.dtype}")
    return E.contiguous(), code


def _params(w: Tensor, b: Tensor) -> Tuple[Tensor, Tensor]:
    """The loss parameters stay float32 whatever the embeddings are."""
    for name, t in (("w", w), ("b", b)):
        if t.dtype != torch.float32:
            raise TypeError(f"{name} must be float32, got {t.dtype}")
    return w.contiguous(), b.contiguous()


def _same_f32c(*ts: Optional[Tensor]) -> None:
    """The staged ops hand raw pointers to fp32 kernels: a half-precision or strided tensor (autocast, a
    slice) would be read and written out of bounds, so refuse it instead of copying (outputs alias)."""
    for t in ts:
        if t is None:
            continue
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise TypeError(f"expected a contiguous float32 CUDA tensor, got {t.dtype}, "
                            f"contiguous={t.is_contiguous()}")
        if not t.is_cuda:
            raise RuntimeError("speaker_embedding_ge2e_loss_b200 runs on CUDA (sm_100a) tensors only; "
                               "there is no CPU fallback")


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _check(rc: int, what: str) -> None:
    """check() for calls that used a cached workspace: a failed call may have left its counters dirty,
    so the cache is dropped and the next call starts from a freshly zeroed buffer."""
    if rc != 0:
        _WS_CACHE.clear()
    check(rc, what)


_WS_CACHE: dict = {}


def _workspace(n_local: int, n_total: int, M: int, D: int, variant: int, precision: int, device):
    """Scratch for fwd_rows / bwd_rows.  Contract of the C ABI: zero on entry; the kernels leave it
    zeroed again, so one buffer per (device, stream, size) is zeroed once and reused (the calls on
    one stream are ordered; another stream gets its own buffer)."""
    nbytes = lib().ge2e_b200_workspace_bytes(n_local, n_total, M, D, variant, precision)
    if nbytes == 0:
        return None, 0
    if torch.cuda.is_current_stream_capturing():
        # inside a capture torch.zeros is only recorded: a cached buffer would be handed to later eager
        # calls without ever having been cleared, and it would pin memory of the graph's private pool
        return torch.zeros(nbytes, dtype=torch.uint8, device=device), nbytes
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream, nbytes)
    ws = _WS_CACHE.get(key)
    if ws is None:
        if len(_WS_CACHE) > 64:
            _WS_CACHE.clear()
        ws = _WS_CACHE[key] = torch.zeros(nbytes, dtype=torch.uint8, device=device)
    return ws, nbytes


# --------------------------------------------------------------------------- single device
class _on_device:
    """`with torch.cuda.device(dev)` only when dev is not already current (the context manager costs
    more host time than the checks below)."""

    def __init__(self, dev):
        self.ctx = None if dev.index is None or dev.index == torch.cuda.current_device() else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def _index_ok(row_index: Optional[Tensor], U: int, dev) -> Optional[Tensor]:
    if row_index is None:
        return None
    if row_index.device != dev or row_index.numel() != U:
        raise ValueError(f"unperm must be a device tensor with {U} entries")
    return row_index.to(torch.int32).contiguous()


def _tc_softmax(N: int, M: int, D: int, variant: int, precision: int) -> bool:
    """True where the softmax loss runs on tensor cores: the forward then also leaves the un-normalised
    dE_hat rows + row_scale (include/ge2e_b200.h, ge2e_b200_fwd_rows) and the backward is one pass."""
    return variant == _lib.SOFTMAX and lib().ge2e_b200_path(N, N, M, D, variant, precision) in (1, 2, 3)


def _fwd_impl(E: Tensor, w: Tensor, b: Tensor, eps: float, variant: int, precision: int, packed: bool,
              row_index: Optional[Tensor] = None, speakers: int = 0, want_grad: bool = True):
    """GE2ELoss.forward (reference s3:19-30) through the C ABI.  ``packed``: the per-call intermediates
    come out of ONE allocation (views); the custom op needs non-aliasing outputs and passes False.
    ``row_index`` (with ``speakers``): E is [U, D] in the embedder's row order and logical row r lives
    at row_index[r] (the trainer's ``embeddings[unperm]``, s4:189-192, folded into the kernels).
    ``want_grad``: a backward will follow (tensor-core softmax path: the forward prepares dE_hat).
    Returns (loss, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale); the last two
    are 1-element placeholders where the path does not use them."""
    _need_cuda(E, w, b)
    (E, ecode), (w, b) = _emb(E), _params(w, b)
    if _lib.planes_need_copy(E.data_ptr(), precision, E.element_size()):
        E = E.clone()
    if row_index is None:
        N, M, D = E.shape
    else:
        U_, D = E.shape
        N, M = speakers, U_ // max(1, speakers)
        if speakers <= 0 or N * M != U_:
            raise ValueError(f"{U_} rows do not split into {speakers} speakers")
    U = N * M
    dev = E.device
    with _on_device(dev):
        fused = want_grad and _tc_softmax(N, M, D, variant, precision)
        nh, ns = (U * D, U) if fused else (1, 1)
        if packed:
            flat = torch.empty(U * D + N * D + 3 * U + 4 + nh + ns, dtype=torch.float32, device=dev)
            o = 0
            e_hat = flat[o:o + U * D].view(U, D); o += U * D
            c_hat = flat[o:o + N * D].view(N, D); o += N * D
            dE_hat = flat[o:o + nh]; o += nh          # 16-byte aligned: U * D and N * D are multiples of 4 here
            cos_diag = flat[o:o + U]; o += U
            row_stat = flat[o:o + U]; o += U
            row_aux = flat[o:o + U]; o += U
            row_scale = flat[o:o + ns]; o += ns
            accum = flat[o:o + 4]
        else:
            accum = torch.empty(4, dtype=torch.float32, device=dev)
            e_hat = torch.empty((U, D), dtype=torch.float32, device=dev)
            c_hat = torch.empty((N, D), dtype=torch.float32, device=dev)
            cos_diag = torch.empty(U, dtype=torch.float32, device=dev)
            row_stat = torch.empty(U, dtype=torch.float32, device=dev)
            row_aux = torch.empty(U, dtype=torch.float32, device=dev)
            dE_hat = torch.empty(nh, dtype=torch.float32, device=dev)
            row_scale = torch.empty(ns, dtype=torch.float32, device=dev)
        if fused:
            dE_hat = dE_hat.view(U, D)
        row_kstar = torch.empty(U if variant == _lib.CONTRAST else 1, dtype=torch.int32, device=dev)
        ws, ws_bytes = _workspace(N, N, M, D, variant, precision, dev)
        rc = lib().ge2e_b200_forward_typed(E.data_ptr(), ecode, _ptr(row_index), N, M, D, w.data_ptr(), b.data_ptr(),
                                           eps, variant, precision, e_hat.data_ptr(), c_hat.data_ptr(),
                                           cos_diag.data_ptr(), row_stat.data_ptr(), row_kstar.data_ptr(),
                                           row_aux.data_ptr(), accum.data_ptr(),
                                           dE_hat.data_ptr() if fused else None,
                                           row_scale.data_ptr() if fused else None, _ptr(ws), ws_bytes, _stream())
    _check(rc, "ge2e_b200_forward")
    return accum[0], e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale


def _bwd_impl(grad_out, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale, eps,
              variant, precision, row_index: Optional[Tensor] = None):
    """loss.backward() (s4:200) through the C ABI.  ``dE_hat`` / ``row_scale``: what the forward prepared
    (1-element placeholders where the path does not use them).  Returns (dE shaped like E, dwdb[2])."""
    _need_cuda(grad_out, E, w, b)
    (E, ecode), (w, b) = _emb(E), _params(w, b)
    g = _f32c(grad_out)
    N, D = c_hat.shape
    U = e_hat.shape[0]
    M = U // N
    _lib.check_backward_shape(M, D)
    dev = E.device
    with _on_device(dev):
        dE = torch.empty_like(E)
        fused = dE_hat.numel() == U * D and _tc_softmax(N, M, D, variant, precision)
        # [accum (4: -, dw, db, -) | dC_hat (N*D) | dE_hat (U*D) unless the forward prepared it]
        scratch = torch.empty(4 + N * D + (0 if fused else U * D), dtype=torch.float32, device=dev)
        dC_ptr = scratch.data_ptr() + 16
        dE_hat_ptr = dE_hat.data_ptr() if fused else dC_ptr + N * D * 4
        ws, ws_bytes = _workspace(N, N, M, D, variant, precision, dev)
        rc = lib().ge2e_b200_backward_typed(E.data_ptr(), ecode, _ptr(row_index), e_hat.data_ptr(), c_hat.data_ptr(),
                                            cos_diag.data_ptr(), row_stat.data_ptr(), row_kstar.data_ptr(),
                                            row_aux.data_ptr(), row_scale.data_ptr() if fused else None, N, M, D,
                                            w.data_ptr(), b.data_ptr(), eps, variant, precision, g.data_ptr(),
                                            dE_hat_ptr, dC_ptr, scratch.data_ptr(), dE.data_ptr(), ecode, _ptr(ws),
                                            ws_bytes, _stream())
    _check(rc, "ge2e_b200_backward")
    return dE, scratch[1:3]


@torch.library.custom_op("ge2e_b200::fwd", mutates_args=())
def ge2e_fwd(E: Tensor, w: Tensor, b: Tensor, eps: float, variant: int,
             precision: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """GE2ELoss.forward as a torch.library op (what torch.compile / export see).  Returns (loss, e_hat,
    c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale); everything after loss is saved for
    the backward."""
    out = _fwd_impl(E, w, b, eps, variant, precision, packed=False)
    return (out[0].clone(),) + out[1:]       # accum[0] is a view of accum: op outputs must not alias


@ge2e_fwd.register_fake
def _(E, w, b, eps, variant, precision):
    N, M, D = E.shape
    U = N * M
    fused = _tc_softmax(N, M, D, variant, precision)
    f32 = torch.float32      # every intermediate is float32 whatever E's element type
    return (E.new_empty((), dtype=f32), E.new_empty((U, D), dtype=f32), E.new_empty((N, D), dtype=f32),
            E.new_empty(U, dtype=f32), E.new_empty(U, dtype=f32),
            E.new_empty(U if variant == _lib.CONTRAST else 1, dtype=torch.int32), E.new_empty(U, dtype=f32),
            E.new_empty((U, D) if fused else (1,), dtype=f32), E.new_empty(U if fused else 1, dtype=f32))


@torch.library.custom_op("ge2e_b200::bwd", mutates_args=())
def ge2e_bwd(grad_out: Tensor, E: Tensor, w: Tensor, b: Tensor, e_hat: Tensor, c_hat: Tensor,
             cos_diag: Tensor, row_stat: Tensor, row_kstar: Tensor, row_aux: Tensor, dE_hat: Tensor,
             row_scale: Tensor, eps: float, variant: int, precision: int) -> Tuple[Tensor, Tensor]:
    """Backward of ge2e_b200::fwd.  Returns (dE[N,M,D], dwdb[2])."""
    dE, dwdb = _bwd_impl(grad_out, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale,
                         eps, variant, precision)
    return dE, dwdb.clone()


@ge2e_bwd.register_fake
def _(grad_out, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale, eps, variant,
      precision):
    return torch.empty_like(E), E.new_empty(2, dtype=torch.float32)


def _fwd_setup(ctx, inputs, output):
    E, w, b, eps, variant, precision = inputs
    _, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale = output
    ctx.save_for_backward(E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale)
    ctx.cfg = (eps, variant, precision)


def _fwd_backward(ctx, g_loss, *_unused):
    E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale = ctx.saved_tensors
    eps, variant, precision = ctx.cfg
    dE, dwdb = ge2e_bwd(g_loss, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale, eps,
                        variant, precision)
    return dE, dwdb[0], dwdb[1], None, None, None


ge2e_fwd.register_autograd(_fwd_backward, setup_context=_fwd_setup)


# --------------------------------------------------------------------------- eager module path
# What `loss = crit(E); loss.backward()` (s4_train_embed_model.py:196-200) costs on the host matters as much
# as the kernels at the reference's batch sizes, so the eager path keeps one _EagerPlan per (device, shape,
# variant, precision): kernel path and workspace size queried once, the intermediates of a step (e_hat,
# c_hat, row statistics, dE_hat, dC_hat: one allocation) taken from a small pool and handed back when the
# autograd node that uses them dies, their pointers pre-bound.  Per step only what ESCAPES to the caller is
# allocated: the 4-float accumulator behind the loss tensor, the one behind dw / db, and dE.
_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _raw_stream(dev_index: int) -> int:
    if _RAW_STREAM is not None:
        return _RAW_STREAM(dev_index)
    return torch.cuda.current_stream(dev_index).cuda_stream


class _StepBufs:
    __slots__ = ("flat", "kstar", "e_hat", "c_hat", "cos_diag", "row_stat", "row_aux", "dE_hat", "row_scale", "dC_hat",
                 "fwd_ptrs", "step_ptrs", "plan", "pooled", "__weakref__")

    def __init__(self, plan, pooled: bool):
        N, M, D, U = plan.N, plan.M, plan.D, plan.U
        dev = plan.device
        ns = U                                  # row_scale: used by the tensor-core softmax paths, required by the ABI
        flat = torch.empty(2 * U * D + 2 * N * D + 3 * U + ns, dtype=torch.float32, device=dev)
        o = 0

        def take(n):
            nonlocal o
            v = flat[o:o + n]
            o += n
            return v
        self.flat = flat
        self.e_hat = take(U * D)
        self.c_hat = take(N * D)
        self.dE_hat = take(U * D)              # forward (tensor-core softmax) or backward scratch
        self.dC_hat = take(N * D)
        self.cos_diag, self.row_stat, self.row_aux = take(U), take(U), take(U)
        self.row_scale = take(ns)
        self.kstar = torch.empty(U if plan.variant == _lib.CONTRAST else 1, dtype=torch.int32, device=dev)
        self.plan, self.pooled = plan, pooled
        self.fwd_ptrs = (self.e_hat.data_ptr(), self.c_hat.data_ptr(), self.cos_diag.data_ptr(), self.row_stat.data_ptr(),
                         self.kstar.data_ptr(), self.row_aux.data_ptr())
        self.step_ptrs = (*self.fwd_ptrs, self.row_scale.data_ptr())


class _EagerPlan:
    __slots__ = ("N", "M", "D", "U", "variant", "precision", "dtype", "device", "dev_index", "path", "fused", "ws_bytes",
                 "free", "one", "free_on", "planes", "bwd_ok")

    def __init__(self, dev, N, M, D, variant, precision, dtype):
        self.N, self.M, self.D, self.U = N, M, D, N * M
        self.variant, self.precision, self.device = variant, precision, dev
        self.dtype = dtype                      # ge2e_dtype code of E and of the dE handed back
        self.dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        h = lib()
        self.path = h.ge2e_b200_path(N, N, M, D, variant, precision)
        self.fused = variant == _lib.SOFTMAX and self.path in (1, 2, 3)
        self.planes = precision in (_lib.FP32_SPLIT, _lib.F16)
        self.bwd_ok = M <= h.ge2e_b200_max_utterances(D)
        # the whole-step entry point (single-kernel step for reference-sized batches) may need more than the stages
        self.ws_bytes = max(h.ge2e_b200_workspace_bytes(N, N, M, D, variant, precision),
                            h.ge2e_b200_step_workspace_bytes(N, M, D, variant, precision))
        self.free = []
        self.free_on = {}
        self.one = torch.ones((), dtype=torch.float32, device=dev)      # upstream gradient of the step run in forward

    def take(self) -> _StepBufs:
        if torch.cuda.is_current_stream_capturing():
            return _StepBufs(self, pooled=False)      # memory of a capture belongs to the graph's pool: never recycled
        return self.free.pop() if self.free else _StepBufs(self, pooled=True)

    def give(self, bufs: _StepBufs) -> None:
        if bufs.pooled and len(self.free) < 4:
            self.free.append(bufs)

    def take_on(self, stream: int) -> _StepBufs:
        """Scratch for a step whose every use is enqueued on `stream` before this returns to the caller: handed
        back at once (give_on) and reused by the next step on the SAME stream, where stream order protects it."""
        if torch.cuda.is_current_stream_capturing():
            return _StepBufs(self, pooled=False)
        q = self.free_on.get(stream)
        return q.pop() if q else _StepBufs(self, pooled=True)

    def give_on(self, bufs: _StepBufs, stream: int) -> None:
        if bufs.pooled:
            if len(self.free_on) > 8:
                self.free_on.clear()
            q = self.free_on.setdefault(stream, [])
            if len(q) < 2:
                q.append(bufs)

    def workspace(self, stream: int):
        if self.ws_bytes == 0:
            return None
        if torch.cuda.is_current_stream_capturing():
            return torch.zeros(self.ws_bytes, dtype=torch.uint8, device=self.device)
        key = (self.dev_index, stream, self.ws_bytes)
        ws = _WS_CACHE.get(key)
        if ws is None:
            if len(_WS_CACHE) > 64:
                _WS_CACHE.clear()
            ws = _WS_CACHE[key] = torch.zeros(self.ws_bytes, dtype=torch.uint8, device=self.device)
        return ws


_EAGER_PLANS: dict = {}
_TORCH_DTYPES = {code: dt for dt, code in _DTYPES.items()}


def _eager_plan(dev, N, M, D, variant, precision, dtype) -> _EagerPlan:
    key = (dev.index, N, M, D, variant, precision, dtype)
    plan = _EAGER_PLANS.get(key)
    if plan is None:
        if len(_EAGER_PLANS) > 32:
            _EAGER_PLANS.clear()
        plan = _EAGER_PLANS[key] = _EagerPlan(dev, N, M, D, variant, precision, dtype)
    return plan


class _Lease:
    """Returns the step's buffers to the pool when the autograd node (ctx) that holds it is collected --
    i.e. when no backward through this forward can happen any more."""
    __slots__ = ("bufs",)

    def __init__(self, bufs):
        self.bufs = bufs

    def __del__(self):
        b = self.bufs
        if b is not None:
            b.plan.give(b)


class _GE2EEager(torch.autograd.Function):
    """ge2e_b200_forward_typed / ge2e_b200_backward_typed without the torch.library dispatch layers
    (which cost ~0.2 ms of host time per step: more than the kernels at every size up to cfg3)."""

    @staticmethod
    def forward(ctx, E, w, b, eps, variant, precision, row_index, speakers):
        if not (E.is_cuda and w.is_cuda and b.is_cuda):
            raise RuntimeError("speaker_embedding_ge2e_loss_b200 runs on CUDA (sm_100a) tensors only; "
                               "there is no CPU fallback")
        (E, ecode), _ = _emb(E), _params(w, b)
        if row_index is None:
            N, M, D = E.shape
        else:
            U_, D = E.shape
            N, M = speakers, U_ // max(1, speakers)
            if speakers <= 0 or N * M != U_:
                raise ValueError(f"{U_} rows do not split into {speakers} speakers")
        dev = E.device
        plan = _eager_plan(dev, N, M, D, variant, precision, ecode)
        if plan.planes and E.data_ptr() % (4 * E.element_size()):
            E = E.clone()           # the fp16-plane kernels read E four elements at a time
        want_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        if want_grad and not plan.bwd_ok:
            _lib.check_backward_shape(M, D)
        if want_grad:
            # A loss somebody will differentiate (s4:196 + s4:200): the WHOLE step now, with upstream gradient 1 --
            # one C call: one kernel for reference-sized batches, prep + ONE persistent step kernel + finalize on
            # the tensor-core paths (instead of a forward and a backward that each cross the grid) -- and backward
            # only scales by the real upstream gradient.  A forward under grad mode that is never differentiated
            # (s4:103) pays for gradients it does not use; wrap it in torch.no_grad() to get the forward kernels.
            with _on_device(dev):
                stream = _raw_stream(plan.dev_index)
                bufs = plan.take_on(stream)
                accum = torch.empty(4, dtype=torch.float32, device=dev)     # escapes as the loss tensor: never pooled
                # the gradient for upstream gradient 1 stays float32: backward rounds g * dE to E's type once, so a
                # loss scale reaches small fp16 gradients before the rounding does
                dE = torch.empty_like(E, dtype=torch.float32)
                ws = plan.workspace(stream)
                rc = lib().ge2e_b200_forward_backward_typed(
                    E.data_ptr(), ecode, _ptr(row_index), N, M, D, w.data_ptr(), b.data_ptr(), eps, variant, precision,
                    plan.one.data_ptr(), *bufs.step_ptrs, accum.data_ptr(), bufs.dE_hat.data_ptr(), bufs.dC_hat.data_ptr(),
                    dE.data_ptr(), _lib.DT_F32, _ptr(ws), plan.ws_bytes, stream)
            _check(rc, "ge2e_b200_forward_backward")
            plan.give_on(bufs, stream)  # the next step on this stream may overwrite them: stream order
            ctx.lease = None
            ctx.cfg = (plan, dE, accum)
            return accum[0]
        with _on_device(dev):
            bufs = plan.take()
            accum = torch.empty(4, dtype=torch.float32, device=dev)     # escapes as the loss tensor: never pooled
            stream = _raw_stream(plan.dev_index)
            ws = plan.workspace(stream)
            fused = False
            rc = lib().ge2e_b200_forward_typed(
                E.data_ptr(), ecode, _ptr(row_index), N, M, D, w.data_ptr(), b.data_ptr(), eps, variant, precision,
                *bufs.fwd_ptrs, accum.data_ptr(), bufs.dE_hat.data_ptr() if fused else None,
                bufs.row_scale.data_ptr() if fused else None, _ptr(ws), plan.ws_bytes, stream)
        _check(rc, "ge2e_b200_forward")
        ctx.save_for_backward(E, w, b)
        ctx.lease = _Lease(bufs)
        ctx.cfg = (eps, variant, precision, plan, fused, row_index, N, M, D)
        return accum[0]

    @staticmethod
    def backward(ctx, g_loss):
        if len(ctx.cfg) == 3:           # the step ran in forward with upstream gradient 1: scale by the real one
            plan, dE1, acc1 = ctx.cfg
            dev = dE1.device
            g = g_loss if (g_loss.dtype == torch.float32 and g_loss.is_cuda) else g_loss.to(dev, torch.float32)
            with _on_device(dev):
                dE = torch.empty_like(dE1, dtype=_TORCH_DTYPES[plan.dtype])
                dwdb = torch.empty(2, dtype=torch.float32, device=dev)      # escapes as dw / db
                rc = lib().ge2e_b200_scale_grads_typed(dE1.data_ptr(), dE.data_ptr(), plan.dtype, dE1.numel(),
                                                       acc1.data_ptr() + 4, dwdb.data_ptr(), g.data_ptr(),
                                                       _raw_stream(plan.dev_index))
            _check(rc, "ge2e_b200_scale_grads_typed")
            return dE, dwdb[0], dwdb[1], None, None, None, None, None
        E, w, b = ctx.saved_tensors
        eps, variant, precision, plan, fused, row_index, N, M, D = ctx.cfg
        bufs = ctx.lease.bufs
        g = g_loss if (g_loss.dtype == torch.float32 and g_loss.is_cuda) else g_loss.to(E.device, torch.float32)
        dev = E.device
        with _on_device(dev):
            dE = torch.empty_like(E)
            accum = torch.empty(4, dtype=torch.float32, device=dev)     # escapes as dw / db: never pooled
            stream = _raw_stream(plan.dev_index)
            ws = plan.workspace(stream)
            rc = lib().ge2e_b200_backward_typed(
                E.data_ptr(), plan.dtype, _ptr(row_index), bufs.e_hat.data_ptr(), bufs.c_hat.data_ptr(),
                bufs.cos_diag.data_ptr(), bufs.row_stat.data_ptr(), bufs.kstar.data_ptr(), bufs.row_aux.data_ptr(),
                bufs.row_scale.data_ptr() if fused else None, N, M, D, w.data_ptr(), b.data_ptr(), eps, variant,
                precision, g.data_ptr(), bufs.dE_hat.data_ptr(), bufs.dC_hat.data_ptr(), accum.data_ptr(), dE.data_ptr(),
                plan.dtype, _ptr(ws), plan.ws_bytes, stream)
        _check(rc, "ge2e_b200_backward_typed")
        return dE, accum[1], accum[2], None, None, None, None, None


# host-only query (a ctypes call): under torch.compile its answer is a constant of the traced graph
_resolve_precision = torch.compiler.assume_constant_result(_lib.resolve_precision)


def ge2e_loss(E: Tensor, w: Tensor, b: Tensor, eps: float = 1e-6, variant: str = "softmax",
              precision: str = "fp32", unperm: Optional[Tensor] = None, speakers: int = 0) -> Tensor:
    """Functional form: differentiable in E, w, b.  Eager calls go through a plain autograd.Function;
    under torch.compile the registered custom ops (same kernels) are used.

    ``unperm`` (with ``speakers`` = N): E is the embedder's output [N*M, D] in shuffled row order and
    the loss is that of ``E[unperm].reshape(N, M, D)`` (s4_train_embed_model.py:189-192); the gather and
    the scatter of its backward happen inside the kernels, dE comes back in E's row order."""
    if unperm is not None:
        if E.dim() != 2:
            raise ValueError(f"with unperm the embeddings must be [N*M, D], got {tuple(E.shape)}")
        if speakers <= 0 or E.shape[0] % speakers != 0 or E.shape[0] // speakers < 2:
            raise ValueError("speakers must divide the number of rows, with M >= 2 utterances per speaker")
        N, vcode = speakers, _lib.VARIANTS[variant]
        pcode = _resolve_precision(precision, N, N, E.shape[0] // N, E.shape[1], vcode)
        if torch.compiler.is_compiling():
            return ge2e_fwd(E[unperm].reshape(N, E.shape[0] // N, E.shape[1]), w, b, float(eps), vcode, pcode)[0]
        idx = _index_ok(unperm, E.shape[0], E.device)
        return _GE2EEager.apply(E, w, b, float(eps), vcode, pcode, idx, speakers)
    if E.dim() != 3:
        raise ValueError(f"embeddings must be [N, M, D], got {tuple(E.shape)}")
    if E.shape[1] < 2:
        raise ValueError("GE2E needs M >= 2 utterances per speaker (the reference divides by M - 1)")
    vcode = _lib.VARIANTS[variant]
    pcode = _resolve_precision(precision, E.shape[0], E.shape[0], E.shape[1], E.shape[2], vcode)
    if torch.compiler.is_compiling():
        return ge2e_fwd(E, w, b, float(eps), vcode, pcode)[0]
    return _GE2EEager.apply(E, w, b, float(eps), vcode, pcode, None, 0)


# --------------------------------------------------------------------------- staged (plain functions)
def prep(E: Tensor, c_hat_local_out: Tensor, precision: int):
    """Stage 1 on the local speakers; writes c_hat into ``c_hat_local_out`` (a slice of the
    all-gather buffer).  Returns (e_hat, cos_diag, accum)."""
    _need_cuda(E, c_hat_local_out)
    E, ecode = _emb(E)
    if _lib.planes_need_copy(E.data_ptr(), precision, E.element_size()):
        E = E.clone()
    _same_f32c(c_hat_local_out)
    n, M, D = E.shape
    dev = E.device
    e_hat = torch.empty((n * M, D), dtype=torch.float32, device=dev)
    cos_diag = torch.empty(n * M, dtype=torch.float32, device=dev)
    accum = torch.empty(4, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = lib().ge2e_b200_prep_typed(E.data_ptr(), ecode, None, n, M, D, precision, e_hat.data_ptr(),
                                        c_hat_local_out.data_ptr(), cos_diag.data_ptr(), accum.data_ptr(), _stream())
    check(rc, "ge2e_b200_prep_typed")
    return e_hat, cos_diag, accum


def fwd_rows(e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant, precision,
             accum, per_row: bool = False, sim: bool = False, want_grad: bool = False):
    """Returns (row_stat, row_kstar, row_aux, per_row, sim, dE_hat, row_scale); the last two are None
    unless ``want_grad`` and the softmax loss runs on tensor cores for this shape (the forward then
    prepares the un-normalised dE_hat: hand both to bwd_rows / bwd_finalize)."""
    _same_f32c(e_hat, c_hat_all, cos_diag, w, b, accum)
    dev = e_hat.device
    U = n_local * M
    fused = (want_grad and variant == _lib.SOFTMAX and not sim
             and lib().ge2e_b200_path(n_local, n_total, M, D, variant, precision) in (1, 2, 3))
    dE_hat = torch.empty((U, D), dtype=torch.float32, device=dev) if fused else None
    row_scale = torch.empty(U, dtype=torch.float32, device=dev) if fused else None
    row_stat = torch.empty(U, dtype=torch.float32, device=dev)
    row_kstar = torch.empty(U if variant == _lib.CONTRAST else 1, dtype=torch.int32, device=dev)
    row_aux = torch.empty(U, dtype=torch.float32, device=dev)
    per = torch.empty(U, dtype=torch.float32, device=dev) if per_row else None
    sim_out = torch.empty((U, n_total), dtype=torch.float32, device=dev) if sim else None
    with torch.cuda.device(dev):
        ws, ws_bytes = _workspace(n_local, n_total, M, D, variant, precision, dev)
        rc = lib().ge2e_b200_fwd_rows(e_hat.data_ptr(), c_hat_all.data_ptr(), cos_diag.data_ptr(), n_local,
                                      n_total, spk_offset, M, D, w.data_ptr(), b.data_ptr(), eps, variant,
                                      precision, row_stat.data_ptr(), row_kstar.data_ptr(), row_aux.data_ptr(),
                                      accum.data_ptr(), _ptr(per), _ptr(sim_out), _ptr(dE_hat), _ptr(row_scale),
                                      _ptr(ws), ws_bytes, _stream())
    _check(rc, "ge2e_b200_fwd_rows")
    return row_stat, row_kstar, row_aux, per, sim_out, dE_hat, row_scale


def bwd_rows(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, n_local, n_total, spk_offset, M, D, w, b,
             eps, variant, precision, grad_out, dE_hat=None, row_scale=None):
    """Returns (dE_hat[U_local, D], dC_hat_partial[n_total, D], dwdb[2]).  ``dE_hat`` / ``row_scale``: what
    fwd_rows(want_grad=True) returned (None: dE_hat is computed here)."""
    _same_f32c(e_hat, c_hat_all, cos_diag, row_stat, row_aux, w, b, grad_out, dE_hat, row_scale)
    dev = e_hat.device
    if dE_hat is None or row_scale is None:
        dE_hat, row_scale = torch.empty((n_local * M, D), dtype=torch.float32, device=dev), None
    scratch = torch.empty(n_total * D + 2, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws, ws_bytes = _workspace(n_local, n_total, M, D, variant, precision, dev)
        rc = lib().ge2e_b200_bwd_rows(e_hat.data_ptr(), c_hat_all.data_ptr(), cos_diag.data_ptr(),
                                      row_stat.data_ptr(), row_kstar.data_ptr(), row_aux.data_ptr(),
                                      _ptr(row_scale), n_local,
                                      n_total, spk_offset, M, D, w.data_ptr(), b.data_ptr(), eps, variant, precision,
                                      grad_out.data_ptr(), dE_hat.data_ptr(), scratch.data_ptr(),
                                      scratch.data_ptr() + n_total * D * 4, _ptr(ws), ws_bytes, _stream())
    _check(rc, "ge2e_b200_bwd_rows")
    return dE_hat, scratch[:n_total * D].view(n_total, D), scratch[n_total * D:]


def bwd_finalize(E, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, w, b, eps, variant, grad_out,
                 row_scale=None):
    """dE in E's element type (fp32, bf16 or fp16), rounded once."""
    E, ecode = _emb(E)
    _same_f32c(dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, w, b, grad_out, row_scale)
    _need_cuda(E)
    n, M, D = E.shape
    dE = torch.empty_like(E)
    with torch.cuda.device(E.device):
        rc = lib().ge2e_b200_bwd_finalize_typed(E.data_ptr(), ecode, None, dE_hat.data_ptr(), dC_hat_local.data_ptr(),
                                                cos_diag.data_ptr(), row_stat.data_ptr(), row_aux.data_ptr(),
                                                _ptr(row_scale), n, M, D, w.data_ptr(), b.data_ptr(), eps, variant,
                                                grad_out.data_ptr(), dE.data_ptr(), ecode, _stream())
    check(rc, "ge2e_b200_bwd_finalize_typed")
    return dE
