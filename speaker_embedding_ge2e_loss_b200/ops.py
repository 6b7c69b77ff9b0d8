"""torch.library custom ops over the C ABI (CUDA only; raises on CPU tensors).

``ge2e_b200::fwd`` / ``ge2e_b200::bwd`` are the single-device ops (``fwd_per_row`` / ``bwd_per_row``: the
per-utterance losses of reduction="none" and their per-row upstream gradient); the staged ops
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


def _cached_workspace(nbytes: int, device, dev_index: int, stream: int) -> Optional[Tensor]:
    """Scratch of the rows kernels.  Contract of the C ABI: zero on entry; the kernels leave it zeroed again, so
    one buffer per (device, stream, size) is zeroed once and reused (the calls on one stream are ordered; another
    stream gets its own buffer)."""
    if nbytes == 0:
        return None
    if torch.cuda.is_current_stream_capturing():
        # inside a capture torch.zeros is only recorded: a cached buffer would be handed to later eager
        # calls without ever having been cleared, and it would pin memory of the graph's private pool
        return torch.zeros(nbytes, dtype=torch.uint8, device=device)
    key = (dev_index, stream, nbytes)
    ws = _WS_CACHE.get(key)
    if ws is None:
        if len(_WS_CACHE) > 64:
            _WS_CACHE.clear()
        ws = _WS_CACHE[key] = torch.zeros(nbytes, dtype=torch.uint8, device=device)
    return ws


def _workspace(n_local: int, n_total: int, M: int, D: int, variant: int, precision: int, device, per_row: bool = False):
    """(workspace, its size) for fwd_rows / bwd_rows and the custom ops, on the current stream.  ``per_row``: also
    large enough for the per-utterance halves of the single-kernel step (what the eager module runs)."""
    nbytes = lib().ge2e_b200_workspace_bytes(n_local, n_total, M, D, variant, precision)
    if per_row:
        nbytes = max(nbytes, lib().ge2e_b200_step_workspace_bytes(n_total, M, D, variant, precision))
    index = device.index if device.index is not None else torch.cuda.current_device()
    return _cached_workspace(nbytes, device, index, torch.cuda.current_stream(device).cuda_stream), nbytes


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


def _forward(per: Optional[Tensor], *args) -> None:
    """ge2e_b200_forward_typed(*args), or with ``per`` the per-utterance losses through
    ge2e_b200_forward_per_row_typed (whose extra pointer sits in front of workspace, size and stream)."""
    if per is None:
        _check(lib().ge2e_b200_forward_typed(*args), "ge2e_b200_forward")
    else:
        _check(lib().ge2e_b200_forward_per_row_typed(*args[:-3], per.data_ptr(), *args[-3:]),
               "ge2e_b200_forward_per_row_typed")


def _fwd_impl(E: Tensor, w: Tensor, b: Tensor, eps: float, variant: int, precision: int, per_row: bool = False):
    """GE2ELoss.forward (reference s3:19-30) through the C ABI, with a backward to follow.  Returns (loss, e_hat,
    c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale); the last two are 1-element placeholders where
    the forward does not prepare them (_lib.prepares_dE_hat).  ``per_row``: the first element is the per-utterance
    losses [N, M] (logical order) instead of their sum."""
    _need_cuda(E, w, b)
    (E, ecode), (w, b) = _emb(E), _params(w, b)
    if _lib.planes_need_copy(E.data_ptr(), precision, E.element_size()):
        E = E.clone()
    N, M, D = E.shape
    U = N * M
    dev = E.device
    with _on_device(dev):
        fused = _lib.prepares_dE_hat(N, N, M, D, variant, precision)
        accum = torch.empty(4, dtype=torch.float32, device=dev)
        e_hat = torch.empty((U, D), dtype=torch.float32, device=dev)
        c_hat = torch.empty((N, D), dtype=torch.float32, device=dev)
        cos_diag = torch.empty(U, dtype=torch.float32, device=dev)
        row_stat = torch.empty(U, dtype=torch.float32, device=dev)
        row_aux = torch.empty(U, dtype=torch.float32, device=dev)
        dE_hat = torch.empty((U, D) if fused else 1, dtype=torch.float32, device=dev)
        row_scale = torch.empty(U if fused else 1, dtype=torch.float32, device=dev)
        row_kstar = torch.empty(U if variant == _lib.CONTRAST else 1, dtype=torch.int32, device=dev)
        per = torch.empty((N, M), dtype=torch.float32, device=dev) if per_row else None
        ws, ws_bytes = _workspace(N, N, M, D, variant, precision, dev, per_row)
        _forward(per, E.data_ptr(), ecode, None, N, M, D, w.data_ptr(), b.data_ptr(), eps, variant, precision,
                 e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(), row_stat.data_ptr(), row_kstar.data_ptr(),
                 row_aux.data_ptr(), accum.data_ptr(), dE_hat.data_ptr() if fused else None,
                 row_scale.data_ptr() if fused else None, _ptr(ws), ws_bytes, _stream())
    return accum[0] if per is None else per, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale


def _bwd_impl(grad_out, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale, eps,
              variant, precision, per_row: bool = False):
    """loss.backward() (s4:200) through the C ABI.  ``dE_hat`` / ``row_scale``: what the forward prepared
    (1-element placeholders where the path does not use them).  ``per_row``: grad_out is the upstream gradient
    of the per-utterance losses, [N, M].  Returns (dE shaped like E, dwdb[2])."""
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
        fused = dE_hat.numel() == U * D and _lib.prepares_dE_hat(N, N, M, D, variant, precision)
        # [accum (4: -, dw, db, -) | dC_hat (N*D) | dE_hat (U*D) unless the forward prepared it]
        scratch = torch.empty(4 + N * D + (0 if fused else U * D), dtype=torch.float32, device=dev)
        dC_ptr = scratch.data_ptr() + 16
        dE_hat_ptr = dE_hat.data_ptr() if fused else dC_ptr + N * D * 4
        ws, ws_bytes = _workspace(N, N, M, D, variant, precision, dev, per_row)
        if per_row and g.numel() != U:
            raise ValueError(f"the upstream gradient of the per-utterance losses needs {U} entries, got {g.numel()}")
        entry = lib().ge2e_b200_backward_per_row_typed if per_row else lib().ge2e_b200_backward_typed
        rc = entry(E.data_ptr(), ecode, None, e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(),
                   row_stat.data_ptr(), row_kstar.data_ptr(), row_aux.data_ptr(), row_scale.data_ptr() if fused else None,
                   N, M, D, w.data_ptr(), b.data_ptr(), eps, variant, precision, g.data_ptr(), dE_hat_ptr, dC_ptr,
                   scratch.data_ptr(), dE.data_ptr(), ecode, _ptr(ws), ws_bytes, _stream())
    _check(rc, "ge2e_b200_backward_per_row_typed" if per_row else "ge2e_b200_backward")
    return dE, scratch[1:3]


@torch.library.custom_op("ge2e_b200::fwd", mutates_args=())
def ge2e_fwd(E: Tensor, w: Tensor, b: Tensor, eps: float, variant: int,
             precision: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """GE2ELoss.forward as a torch.library op (what torch.compile / export see).  Returns (loss, e_hat,
    c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale); everything after loss is saved for
    the backward."""
    out = _fwd_impl(E, w, b, eps, variant, precision)
    return (out[0].clone(),) + out[1:]       # accum[0] is a view of accum: op outputs must not alias


def _fake_fwd(E, variant, precision, loss_shape):
    """Outputs of _fwd_impl, for the fakes of ge2e_b200::fwd and ge2e_b200::fwd_per_row."""
    N, M, D = E.shape
    U = N * M
    fused = _lib.prepares_dE_hat(N, N, M, D, variant, precision)
    f32 = torch.float32      # every intermediate is float32 whatever E's element type
    return (E.new_empty(loss_shape, dtype=f32), E.new_empty((U, D), dtype=f32), E.new_empty((N, D), dtype=f32),
            E.new_empty(U, dtype=f32), E.new_empty(U, dtype=f32),
            E.new_empty(U if variant == _lib.CONTRAST else 1, dtype=torch.int32), E.new_empty(U, dtype=f32),
            E.new_empty((U, D) if fused else (1,), dtype=f32), E.new_empty(U if fused else 1, dtype=f32))


def _fake_bwd(grad, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale, eps, variant,
              precision):
    return torch.empty_like(E), E.new_empty(2, dtype=torch.float32)


@ge2e_fwd.register_fake
def _(E, w, b, eps, variant, precision):
    return _fake_fwd(E, variant, precision, ())


@torch.library.custom_op("ge2e_b200::bwd", mutates_args=())
def ge2e_bwd(grad_out: Tensor, E: Tensor, w: Tensor, b: Tensor, e_hat: Tensor, c_hat: Tensor,
             cos_diag: Tensor, row_stat: Tensor, row_kstar: Tensor, row_aux: Tensor, dE_hat: Tensor,
             row_scale: Tensor, eps: float, variant: int, precision: int) -> Tuple[Tensor, Tensor]:
    """Backward of ge2e_b200::fwd.  Returns (dE[N,M,D], dwdb[2])."""
    dE, dwdb = _bwd_impl(grad_out, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale,
                         eps, variant, precision)
    return dE, dwdb.clone()


ge2e_bwd.register_fake(_fake_bwd)


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


@torch.library.custom_op("ge2e_b200::fwd_per_row", mutates_args=())
def ge2e_fwd_per_row(E: Tensor, w: Tensor, b: Tensor, eps: float, variant: int,
                     precision: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """ge2e_b200::fwd with the per-utterance losses [N, M] (reduction="none") in place of their sum."""
    return _fwd_impl(E, w, b, eps, variant, precision, per_row=True)


@ge2e_fwd_per_row.register_fake
def _(E, w, b, eps, variant, precision):
    return _fake_fwd(E, variant, precision, (E.shape[0], E.shape[1]))


@torch.library.custom_op("ge2e_b200::bwd_per_row", mutates_args=())
def ge2e_bwd_per_row(grad_rows: Tensor, E: Tensor, w: Tensor, b: Tensor, e_hat: Tensor, c_hat: Tensor,
                     cos_diag: Tensor, row_stat: Tensor, row_kstar: Tensor, row_aux: Tensor, dE_hat: Tensor,
                     row_scale: Tensor, eps: float, variant: int, precision: int) -> Tuple[Tensor, Tensor]:
    """Backward of ge2e_b200::fwd_per_row for the upstream gradient grad_rows[N, M].  Returns (dE[N,M,D], dwdb[2])."""
    dE, dwdb = _bwd_impl(grad_rows.contiguous(), E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat,
                         row_scale, eps, variant, precision, per_row=True)
    return dE, dwdb.clone()


ge2e_bwd_per_row.register_fake(_fake_bwd)


def _fwd_per_row_backward(ctx, g_rows, *_unused):
    E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale = ctx.saved_tensors
    eps, variant, precision = ctx.cfg
    dE, dwdb = ge2e_bwd_per_row(g_rows.to(torch.float32), E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux,
                                dE_hat, row_scale, eps, variant, precision)
    return dE, dwdb[0], dwdb[1], None, None, None


ge2e_fwd_per_row.register_autograd(_fwd_per_row_backward, setup_context=_fwd_setup)


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
    __slots__ = ("N", "M", "D", "U", "variant", "precision", "dtype", "device", "dev_index", "fused", "ws_bytes",
                 "free", "one", "free_on", "bwd_ok")

    def __init__(self, dev, N, M, D, variant, precision, dtype):
        self.N, self.M, self.D, self.U = N, M, D, N * M
        self.variant, self.precision, self.device = variant, precision, dev
        self.dtype = dtype                      # ge2e_dtype code of E and of the dE handed back
        self.dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        h = lib()
        self.fused = _lib.prepares_dE_hat(N, N, M, D, variant, precision)
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
        return _cached_workspace(self.ws_bytes, self.device, self.dev_index, stream)


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


def _eager_setup(E, w, b, variant, precision, row_index, speakers, want_grad):
    """The checks of an eager call and its plan.  E is [N, M, D], or [N*M, D] in the embedder's row order with
    ``row_index`` and ``speakers`` = N.  Returns (E contiguous, its ge2e_dtype code, plan)."""
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
    plan = _eager_plan(E.device, N, M, D, variant, precision, ecode)
    if _lib.planes_need_copy(E.data_ptr(), precision, E.element_size()):
        E = E.clone()
    if want_grad and not plan.bwd_ok:
        _lib.check_backward_shape(M, D)
    return E, ecode, plan


class _GE2EEager(torch.autograd.Function):
    """The summed loss of inputs that require grad, through ge2e_b200_forward_backward_typed without the
    torch.library dispatch layers (which cost ~0.2 ms of host time per step: more than the kernels at every size up
    to cfg3).  A loss somebody will differentiate (s4:196 + s4:200): the WHOLE step runs in forward, with upstream
    gradient 1 -- one C call: one kernel for reference-sized batches, prep + ONE persistent step kernel + finalize on
    the tensor-core paths (instead of a forward and a backward that each cross the grid) -- and backward only scales
    by the real upstream gradient.  A forward that is never differentiated (s4:103) pays for gradients it does not
    use, under torch.no_grad() too: the choice follows requires_grad of E, w and b, not the grad mode."""

    @staticmethod
    def forward(ctx, E, w, b, eps, variant, precision, row_index, speakers):
        E, ecode, plan = _eager_setup(E, w, b, variant, precision, row_index, speakers, True)
        dev = E.device
        with _on_device(dev):
            stream = _raw_stream(plan.dev_index)
            bufs = plan.take_on(stream)
            accum = torch.empty(4, dtype=torch.float32, device=dev)     # escapes as the loss tensor: never pooled
            # the gradient for upstream gradient 1 stays float32: backward rounds g * dE to E's type once, so a
            # loss scale reaches small fp16 gradients before the rounding does
            dE = torch.empty_like(E, dtype=torch.float32)
            ws = plan.workspace(stream)
            rc = lib().ge2e_b200_forward_backward_typed(
                E.data_ptr(), ecode, _ptr(row_index), plan.N, plan.M, plan.D, w.data_ptr(), b.data_ptr(), eps, variant,
                precision, plan.one.data_ptr(), *bufs.step_ptrs, accum.data_ptr(), bufs.dE_hat.data_ptr(),
                bufs.dC_hat.data_ptr(), dE.data_ptr(), _lib.DT_F32, _ptr(ws), plan.ws_bytes, stream)
        _check(rc, "ge2e_b200_forward_backward")
        plan.give_on(bufs, stream)  # the next step on this stream may overwrite them: stream order
        ctx.cfg = (plan, dE, accum)
        return accum[0]

    @staticmethod
    def backward(ctx, g_loss):
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


class _GE2EStaged(torch.autograd.Function):
    """The staged pipeline: forward kernels now (ge2e_b200_forward_typed, or ge2e_b200_forward_per_row_typed for the
    per-utterance losses L[N, M] in logical order), backward kernels in backward.  It serves reduction="none", whose
    upstream gradient is unknown when the forward runs, and the summed loss when no input requires grad.  Where a
    gradient will follow, the tensor-core softmax paths also prepare dE_hat / row_scale in the forward."""

    @staticmethod
    def forward(ctx, E, w, b, eps, variant, precision, row_index, speakers, per_row):
        want_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        E, ecode, plan = _eager_setup(E, w, b, variant, precision, row_index, speakers, want_grad)
        fused = want_grad and plan.fused
        dev = E.device
        with _on_device(dev):
            bufs = plan.take()
            accum = torch.empty(4, dtype=torch.float32, device=dev)     # escapes as the loss tensor: never pooled
            per = torch.empty((plan.N, plan.M), dtype=torch.float32, device=dev) if per_row else None   # escapes
            stream = _raw_stream(plan.dev_index)
            ws = plan.workspace(stream)
            _forward(per, E.data_ptr(), ecode, _ptr(row_index), plan.N, plan.M, plan.D, w.data_ptr(), b.data_ptr(), eps,
                     variant, precision, *bufs.fwd_ptrs, accum.data_ptr(), bufs.dE_hat.data_ptr() if fused else None,
                     bufs.row_scale.data_ptr() if fused else None, _ptr(ws), plan.ws_bytes, stream)
        ctx.save_for_backward(E, w, b)
        ctx.lease = _Lease(bufs)
        ctx.cfg = (eps, variant, precision, plan, fused, row_index)
        return accum[0] if per is None else per

    @staticmethod
    def backward(ctx, g_per):
        # reduction="none" only: a summed loss comes here only when no input requires grad, and then has no grad_fn
        E, w, b = ctx.saved_tensors
        eps, variant, precision, plan, fused, row_index = ctx.cfg
        bufs = ctx.lease.bufs
        dev = E.device
        # one float32 per utterance row, contiguous: `per.sum().backward()` hands over an expanded (stride-0) ones
        g = g_per.to(dev, torch.float32).contiguous()
        with _on_device(dev):
            dE = torch.empty_like(E)
            accum = torch.empty(4, dtype=torch.float32, device=dev)     # escapes as dw / db: never pooled
            stream = _raw_stream(plan.dev_index)
            ws = plan.workspace(stream)
            rc = lib().ge2e_b200_backward_per_row_typed(
                E.data_ptr(), plan.dtype, _ptr(row_index), bufs.e_hat.data_ptr(), bufs.c_hat.data_ptr(),
                bufs.cos_diag.data_ptr(), bufs.row_stat.data_ptr(), bufs.kstar.data_ptr(), bufs.row_aux.data_ptr(),
                bufs.row_scale.data_ptr() if fused else None, plan.N, plan.M, plan.D, w.data_ptr(), b.data_ptr(), eps,
                variant, precision, g.data_ptr(), bufs.dE_hat.data_ptr(), bufs.dC_hat.data_ptr(), accum.data_ptr(),
                dE.data_ptr(), plan.dtype, _ptr(ws), plan.ws_bytes, stream)
        _check(rc, "ge2e_b200_backward_per_row_typed")
        return dE, accum[1], accum[2], None, None, None, None, None, None


def _apply(E, w, b, eps, variant, precision, row_index, speakers, per_row):
    # the test of ctx.needs_input_grad, made before apply: requires_grad, whatever the grad mode
    if per_row or not (E.requires_grad or w.requires_grad or b.requires_grad):
        return _GE2EStaged.apply(E, w, b, eps, variant, precision, row_index, speakers, per_row)
    return _GE2EEager.apply(E, w, b, eps, variant, precision, row_index, speakers)


# host-only query (a ctypes call): under torch.compile its answer is a constant of the traced graph
_resolve_precision = torch.compiler.assume_constant_result(_lib.resolve_precision)


REDUCTIONS = ("sum", "mean", "none")


def ge2e_loss(E: Tensor, w: Tensor, b: Tensor, eps: float = 1e-6, variant: str = "softmax",
              precision: str = "fp32", unperm: Optional[Tensor] = None, speakers: int = 0, *,
              reduction: str = "sum") -> Tensor:
    """Functional form: differentiable in E, w, b.  Eager calls go through a plain autograd.Function;
    under torch.compile the registered custom ops (same kernels) are used.

    ``unperm`` (with ``speakers`` = N): E is the embedder's output [N*M, D] in shuffled row order and
    the loss is that of ``E[unperm].reshape(N, M, D)`` (s4_train_embed_model.py:189-192); the gather and
    the scatter of its backward happen inside the kernels, dE comes back in E's row order.

    ``reduction``: "sum" (the reference's 0-dim loss), "mean" (the sum over N*M) or "none": the per-utterance
    losses L[N, M] as float32 in logical [speaker][utterance] order (calc_loss's per_embedding_loss, s3:121),
    differentiable for any upstream gradient g[N, M]."""
    if reduction not in REDUCTIONS:
        raise ValueError(f"reduction must be one of {REDUCTIONS}, got {reduction!r}")
    loss = _ge2e_loss(E, w, b, eps, variant, precision, unperm, speakers, reduction == "none")
    if reduction == "mean":
        return loss / (E.shape[0] if unperm is not None else E.shape[0] * E.shape[1])
    return loss


def _ge2e_loss(E, w, b, eps, variant, precision, unperm, speakers, per_row: bool) -> Tensor:
    if unperm is not None:
        if E.dim() != 2:
            raise ValueError(f"with unperm the embeddings must be [N*M, D], got {tuple(E.shape)}")
        if speakers <= 0 or E.shape[0] % speakers != 0 or E.shape[0] // speakers < 2:
            raise ValueError("speakers must divide the number of rows, with M >= 2 utterances per speaker")
        N, vcode = speakers, _lib.VARIANTS[variant]
        pcode = _resolve_precision(precision, N, N, E.shape[0] // N, E.shape[1], vcode)
        if torch.compiler.is_compiling():
            op = ge2e_fwd_per_row if per_row else ge2e_fwd
            return op(E[unperm].reshape(N, E.shape[0] // N, E.shape[1]), w, b, float(eps), vcode, pcode)[0]
        idx = _index_ok(unperm, E.shape[0], E.device)
        return _apply(E, w, b, float(eps), vcode, pcode, idx, speakers, per_row)
    if E.dim() != 3:
        raise ValueError(f"embeddings must be [N, M, D], got {tuple(E.shape)}")
    if E.shape[1] < 2:
        raise ValueError("GE2E needs M >= 2 utterances per speaker (the reference divides by M - 1)")
    vcode = _lib.VARIANTS[variant]
    pcode = _resolve_precision(precision, E.shape[0], E.shape[0], E.shape[1], E.shape[2], vcode)
    if torch.compiler.is_compiling():
        return (ge2e_fwd_per_row if per_row else ge2e_fwd)(E, w, b, float(eps), vcode, pcode)[0]
    return _apply(E, w, b, float(eps), vcode, pcode, None, 0, per_row)


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
    fused = want_grad and not sim and _lib.prepares_dE_hat(n_local, n_total, M, D, variant, precision)
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
    fwd_rows(want_grad=True) returned (None: dE_hat is computed here).  ``grad_out``: the scalar upstream gradient,
    or one per local utterance row (U_local elements, logical order: the per-utterance losses)."""
    _same_f32c(e_hat, c_hat_all, cos_diag, row_stat, row_aux, w, b, grad_out, dE_hat, row_scale)
    dev = e_hat.device
    per_row = _per_row_grad(grad_out, n_local * M)
    if dE_hat is None or row_scale is None:
        dE_hat, row_scale = torch.empty((n_local * M, D), dtype=torch.float32, device=dev), None
    scratch = torch.empty(n_total * D + 2, dtype=torch.float32, device=dev)
    entry = "ge2e_b200_bwd_rows_per_row" if per_row else "ge2e_b200_bwd_rows"
    with torch.cuda.device(dev):
        ws, ws_bytes = _workspace(n_local, n_total, M, D, variant, precision, dev)
        rc = getattr(lib(), entry)(e_hat.data_ptr(), c_hat_all.data_ptr(), cos_diag.data_ptr(),
                                   row_stat.data_ptr(), row_kstar.data_ptr(), row_aux.data_ptr(),
                                   _ptr(row_scale), n_local,
                                   n_total, spk_offset, M, D, w.data_ptr(), b.data_ptr(), eps, variant, precision,
                                   grad_out.data_ptr(), dE_hat.data_ptr(), scratch.data_ptr(),
                                   scratch.data_ptr() + n_total * D * 4, _ptr(ws), ws_bytes, _stream())
    _check(rc, entry)
    return dE_hat, scratch[:n_total * D].view(n_total, D), scratch[n_total * D:]


def _per_row_grad(grad_out: Tensor, U: int) -> bool:
    """True for an upstream gradient with one entry per utterance row, False for a scalar (M >= 2: U > 1)."""
    if grad_out.numel() == 1:
        return False
    if grad_out.numel() != U:
        raise ValueError(f"the upstream gradient needs 1 or {U} entries (one per utterance row), got {grad_out.numel()}")
    return True


def bwd_finalize(E, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, w, b, eps, variant, grad_out,
                 row_scale=None):
    """dE in E's element type (fp32, bf16 or fp16), rounded once.  ``grad_out``: scalar or per row, as in bwd_rows."""
    E, ecode = _emb(E)
    _same_f32c(dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, w, b, grad_out, row_scale)
    _need_cuda(E)
    n, M, D = E.shape
    entry = "ge2e_b200_bwd_finalize_per_row_typed" if _per_row_grad(grad_out, n * M) else "ge2e_b200_bwd_finalize_typed"
    dE = torch.empty_like(E)
    with torch.cuda.device(E.device):
        rc = getattr(lib(), entry)(E.data_ptr(), ecode, None, dE_hat.data_ptr(), dC_hat_local.data_ptr(),
                                   cos_diag.data_ptr(), row_stat.data_ptr(), row_aux.data_ptr(),
                                   _ptr(row_scale), n, M, D, w.data_ptr(), b.data_ptr(), eps, variant,
                                   grad_out.data_ptr(), dE.data_ptr(), ecode, _stream())
    check(rc, entry)
    return dE
