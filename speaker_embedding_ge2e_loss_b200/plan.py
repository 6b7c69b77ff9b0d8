"""Pre-planned GE2E step: every buffer allocated once, fwd+bwd issued as bare C-ABI calls.

``GE2ELoss`` / ``ge2e_loss`` go through ``torch.library`` + autograd, which costs tens of
microseconds of host time per call -- more than the kernels themselves at the repo's batch sizes.
A plan is the launch-latency-free form of the same step (reference call sequence
s4_train_embed_model.py:196-200: ``loss = ge2e_loss(E); loss.backward()``): the library never
allocates or synchronises, so ``step()`` is CUDA-graph capturable (``capture()``).
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, lib
from .ops import _DTYPES


class GE2EPlan:
    def __init__(self, N: int, M: int, D: int, variant: str = "softmax", precision: str = "fp32",
                 eps: float = 1e-6, device=None, sgd=None, dtype: torch.dtype = torch.float32, reduction: str = "sum"):
        """``sgd=(lr, max_norm)``: every step ends with the trainer's tail for the two loss parameters
        (clip_grad_norm_ on (w, b) + plain SGD, s4_train_embed_model.py:202-203) as one more kernel,
        updating the ``w`` / ``b`` passed to ``step`` in place.  ``dtype``: element type of the embeddings
        ``step`` takes (float32, bfloat16 or float16); ``.dE`` has it too, everything else is float32.

        ``reduction="none"``: per-utterance losses.  The forward writes ``.per_row`` ([N, M] float32, logical
        order; ``.loss`` is their sum) and the backward (``backward()``) differentiates sum_r grad_rows[r] L_r with
        ``.grad_rows`` ([N, M] float32, initialised to ones), read when the backward runs -- so a caller can
        weight or mask utterances from ``per_row`` on the device between a captured forward and a captured
        backward.  On the single-kernel step's shapes each half is one kernel."""
        if dtype not in _DTYPES:
            raise TypeError(f"dtype must be float32, bfloat16 or float16, got {dtype}")
        if reduction not in ("sum", "none"):
            raise ValueError(f"GE2EPlan reduction must be 'sum' or 'none', got {reduction!r}")
        self.reduction = reduction
        self.dtype, self._dtype_code = dtype, _DTYPES[dtype]
        self.sgd = None if sgd is None else (float(sgd[0]), float(sgd[1]))
        if M < 2:
            raise ValueError("GE2E needs M >= 2 utterances per speaker")
        self.N, self.M, self.D = N, M, D
        self.variant = _lib.VARIANTS[variant]
        self.eps = float(eps)
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("speaker_embedding_ge2e_loss_b200 runs on CUDA (sm_100a) only; no CPU fallback")
        with torch.cuda.device(self.device):
            self.precision = _lib.resolve_precision(precision, N, N, M, D, self.variant)
        U, dev, f32 = N * M, self.device, torch.float32
        # 0 SIMT fp32, 1 tcgen05 TF32, 2 tcgen05 split fp16 planes (fp32-class)
        self.path = lib().ge2e_b200_path(N, N, M, D, self.variant, self.precision)
        self.e_hat = torch.empty((U, D), dtype=f32, device=dev)
        self.c_hat = torch.empty((N, D), dtype=f32, device=dev)
        self.cos_diag = torch.empty(U, dtype=f32, device=dev)
        self.row_stat = torch.empty(U, dtype=f32, device=dev)
        self.row_kstar = torch.empty(U, dtype=torch.int32, device=dev)
        self.row_aux = torch.empty(U, dtype=f32, device=dev)
        self.dE_hat = torch.empty((U, D), dtype=f32, device=dev)
        self.row_scale = torch.empty(U, dtype=f32, device=dev)   # tensor-core softmax path: factor of the dE_hat rows
        self.dC_hat = torch.empty((N, D), dtype=f32, device=dev)
        self._accum = torch.empty(4, dtype=f32, device=dev)      # {loss, dw, db, -}: zeroed by prep every step
        self.dE = torch.empty((N, M, D), dtype=dtype, device=dev)
        self.grad_out = torch.ones((), dtype=f32, device=dev)
        nbytes = lib().ge2e_b200_step_workspace_bytes(N, M, D, self.variant, self.precision)
        self._ws = torch.zeros(max(nbytes, 1), dtype=torch.uint8, device=dev)   # zero once: the kernels restore it
        # 1: the reference-sized batch runs fwd+bwd as ONE kernel (ge2e_b200_forward_backward)
        self.single_kernel = lib().ge2e_b200_step_launches(N, M, D, self.variant, self.precision) == 1
        self._bwd_ok = M <= lib().ge2e_b200_max_utterances(D)
        self._ws_bytes = nbytes
        self.loss, self.dw, self.db = self._accum[0], self._accum[1], self._accum[2]
        self._graph = None
        if reduction == "none":
            self.per_row = torch.empty((N, M), dtype=f32, device=dev)
            self.grad_rows = torch.ones((N, M), dtype=f32, device=dev)
            # tensor-core softmax: the forward also leaves the un-normalised dE_hat rows + row_scale
            self._scaled = _lib.prepares_dE_hat(N, N, M, D, self.variant, self.precision)
        self._fwd_E = None      # data_ptr of the last forward's E (reduction="none": what backward() differentiates)

    def step(self, E: torch.Tensor, w: torch.Tensor, b: torch.Tensor, backward: bool = True) -> None:
        """Enqueue fwd (+ bwd) on the current stream.  Results land in .loss/.dE/.dw/.db (and .per_row with
        reduction="none", whose backward is ``backward()``)."""
        if E.dtype != self.dtype:
            raise TypeError(f"GE2EPlan was built for {self.dtype} embeddings, got {E.dtype}")
        assert E.is_cuda and E.is_contiguous() and tuple(E.shape) == (self.N, self.M, self.D)
        h, N, M, D, dt = lib(), self.N, self.M, self.D, self._dtype_code
        if _lib.planes_need_copy(E.data_ptr(), self.precision, E.element_size()):
            # a plan copies nothing behind the caller's back (its steps are captured into graphs)
            raise ValueError("GE2EPlan: the fp16-plane precisions need a 16-byte-aligned E (8-byte for bfloat16 / "
                             "float16); this one sits at an "
                             "offset of its storage -- pass E.clone(), or build the plan with precision='fp32_simt'")
        if backward and not self._bwd_ok:
            _lib.check_backward_shape(M, D)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._ws.data_ptr() if self._ws_bytes else None
        if self.reduction == "none":
            rc = h.ge2e_b200_forward_per_row_typed(
                E.data_ptr(), dt, None, N, M, D, w.data_ptr(), b.data_ptr(), self.eps, self.variant, self.precision,
                self.e_hat.data_ptr(), self.c_hat.data_ptr(), self.cos_diag.data_ptr(), self.row_stat.data_ptr(),
                self.row_kstar.data_ptr(), self.row_aux.data_ptr(), self._accum.data_ptr(),
                self.dE_hat.data_ptr() if self._scaled else None, self.row_scale.data_ptr() if self._scaled else None,
                self.per_row.data_ptr(), ws, self._ws_bytes, stream)
            check(rc, "ge2e_b200_forward_per_row_typed")
            self._fwd_E = E.data_ptr()
            if backward:
                self.backward(E, w, b)
            return
        if backward:
            accum_ptr = self._accum.data_ptr()
            rc = h.ge2e_b200_forward_backward_typed(E.data_ptr(), dt, None, N, M, D, w.data_ptr(), b.data_ptr(),
                                                    self.eps, self.variant, self.precision, self.grad_out.data_ptr(),
                                                    self.e_hat.data_ptr(), self.c_hat.data_ptr(),
                                                    self.cos_diag.data_ptr(), self.row_stat.data_ptr(),
                                                    self.row_kstar.data_ptr(), self.row_aux.data_ptr(),
                                                    self.row_scale.data_ptr(), accum_ptr, self.dE_hat.data_ptr(),
                                                    self.dC_hat.data_ptr(), self.dE.data_ptr(), dt, ws, self._ws_bytes,
                                                    stream)
            check(rc, "ge2e_b200_forward_backward_typed")
            self._sgd_tail(w, b, stream)
            return
        rc = h.ge2e_b200_forward_typed(E.data_ptr(), dt, None, N, M, D, w.data_ptr(), b.data_ptr(), self.eps,
                                       self.variant, self.precision, self.e_hat.data_ptr(), self.c_hat.data_ptr(),
                                       self.cos_diag.data_ptr(), self.row_stat.data_ptr(), self.row_kstar.data_ptr(),
                                       self.row_aux.data_ptr(), self._accum.data_ptr(), None, None, ws, self._ws_bytes,
                                       stream)
        check(rc, "ge2e_b200_forward_typed")

    def _sgd_tail(self, w: torch.Tensor, b: torch.Tensor, stream: int) -> None:
        if self.sgd is not None:
            accum_ptr = self._accum.data_ptr()
            rc = lib().ge2e_b200_scale_bias_sgd(w.data_ptr(), b.data_ptr(), accum_ptr + 4, accum_ptr + 8, self.sgd[1],
                                                self.sgd[0], None, stream)
            check(rc, "ge2e_b200_scale_bias_sgd")

    def backward(self, E: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> None:
        """reduction="none": enqueue the backward of the last forward (``step(E, w, b, backward=False)``) for the
        upstream gradient ``.grad_rows`` on the current stream, then the ``sgd=`` tail.  ``E`` is that forward's
        batch.  Results land in .dE/.dw/.db."""
        if self.reduction != "none":
            raise RuntimeError("GE2EPlan.backward() is the per-utterance backward of a reduction='none' plan; "
                               "a 'sum' plan runs its backward inside step()")
        if self._fwd_E is None:
            raise RuntimeError("GE2EPlan.backward() before any forward: call step(E, w, b, backward=False) first")
        if E.data_ptr() != self._fwd_E:
            raise ValueError("GE2EPlan.backward() takes the E of the last forward")
        if not self._bwd_ok:
            _lib.check_backward_shape(self.M, self.D)
        N, M, D, dt = self.N, self.M, self.D, self._dtype_code
        stream = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._ws.data_ptr() if self._ws_bytes else None
        rc = lib().ge2e_b200_backward_per_row_typed(
            E.data_ptr(), dt, None, self.e_hat.data_ptr(), self.c_hat.data_ptr(), self.cos_diag.data_ptr(),
            self.row_stat.data_ptr(), self.row_kstar.data_ptr(), self.row_aux.data_ptr(),
            self.row_scale.data_ptr() if self._scaled else None, N, M, D, w.data_ptr(), b.data_ptr(), self.eps,
            self.variant, self.precision, self.grad_rows.data_ptr(), self.dE_hat.data_ptr(), self.dC_hat.data_ptr(),
            self._accum.data_ptr(), self.dE.data_ptr(), dt, ws, self._ws_bytes, stream)
        check(rc, "ge2e_b200_backward_per_row_typed")
        self._sgd_tail(w, b, stream)

    def _capture(self, enqueue, steps: int):
        """(graph of ``steps`` calls enqueue(k), library launches per call); one eager call first as warm-up."""
        with torch.cuda.device(self.device):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                enqueue(0)                              # warm-up: lazy func attributes, module load
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            before = lib().ge2e_b200_launch_count()
            with torch.cuda.graph(g):
                for k in range(steps):
                    enqueue(k)
            return g, (lib().ge2e_b200_launch_count() - before) // max(1, steps)

    def capture_backward(self, E: torch.Tensor, w: torch.Tensor, b: torch.Tensor):
        """reduction="none": ``backward(E, w, b)`` as a CUDA graph of its own (``.replay()``), to replay after a
        forward graph (``capture(E, w, b, backward=False)``) with ``grad_rows`` set in between.  Records the
        library kernels it launches in ``backward_launches``."""
        g, self.backward_launches = self._capture(lambda k: self.backward(E, w, b), 1)
        return g

    def capture(self, E, w: torch.Tensor, b: torch.Tensor, backward: bool = True, steps: int = 1):
        """Capture ``steps`` consecutive steps into one CUDA graph bound to these tensors; returns the
        graph (``.replay()``).  ``E`` is one batch or a list of batches the steps rotate over.  Also
        records how many of the library's kernels one step launches."""
        batches = list(E) if isinstance(E, (list, tuple)) else [E]
        g, self.launches_per_step = self._capture(lambda k: self.step(batches[k % len(batches)], w, b, backward), steps)
        self._graph = g
        return g


class ShardedGE2EPlan:
    """Speaker-sharded fwd+bwd (one process per GPU) with persistent buffers, the C-ABI stages and the
    three NCCL collectives enqueued back to back so that the whole step can be captured in one CUDA
    graph: prep -> all-gather(c_hat) -> step_rows (forward rows + backward rows: ONE tensor-core kernel for
    the softmax loss) -> reduce-scatter(dC_hat) -> all-reduce({loss, dw, db}) || bwd_finalize.  Upstream gradient = 1 (``loss.backward()``).
    Results: ``.loss`` (global), ``.dE`` (this rank's rows), ``.dw`` / ``.db`` (global)."""

    def __init__(self, n_local: int, n_total: int, spk_offset: int, M: int, D: int, variant: str = "softmax",
                 precision: str = "tf32", eps: float = 1e-6, group=None, device=None, peer_memory="auto"):
        """``peer_memory``: "auto" (default) / True / False.  Where the softmax loss runs on tensor cores and the
        ranks of ``group`` can map each other's memory (one NVLink / NVSwitch domain, <= 8 ranks, n_local a
        multiple of 128), the two exchange steps are done by the kernels themselves over peer memory
        (``torch.distributed._symmetric_memory`` buffers): the all-gather of ``c_hat`` is a store of this rank's
        slice into every peer (``ge2e_b200_peer_publish``), the reduce-scatter of ``dC_hat`` is the step
        kernel's centroid pass adding its accumulator tiles straight into the owner rank's rows
        (``ge2e_b200_step_rows_peers``); two cross-rank barriers replace the two NCCL collectives.  Otherwise
        (or with ``peer_memory=False``) the step uses all_gather_into_tensor / reduce_scatter_tensor.
        All ranks must construct the plan collectively (the buffers are rendezvoused)."""
        import torch.distributed as dist
        self.dist = dist
        self.group = group if group is not None else dist.group.WORLD
        self.n_local, self.n_total, self.spk_offset, self.M, self.D = n_local, n_total, spk_offset, M, D
        self.variant = _lib.VARIANTS[variant]
        self.eps = float(eps)
        self.device = torch.device(device if device is not None else "cuda")
        _lib.check_backward_shape(M, D)
        with torch.cuda.device(self.device):
            self.precision = _lib.resolve_precision(precision, n_local, n_total, M, D, self.variant)
        U, dev, f32 = n_local * M, self.device, torch.float32
        self.e_hat = torch.empty((U, D), dtype=f32, device=dev)
        self.c_hat_all = torch.empty((n_total, D), dtype=f32, device=dev)      # (replaced below in peer-memory mode)
        self.c_hat_mine = self.c_hat_all[spk_offset:spk_offset + n_local]
        self.cos_diag = torch.empty(U, dtype=f32, device=dev)
        self.row_stat = torch.empty(U, dtype=f32, device=dev)
        self.row_kstar = torch.empty(U, dtype=torch.int32, device=dev)
        self.row_aux = torch.empty(U, dtype=f32, device=dev)
        self.dE_hat = torch.empty((U, D), dtype=f32, device=dev)
        self.row_scale = torch.empty(U, dtype=f32, device=dev)
        self.path = lib().ge2e_b200_path(n_local, n_total, M, D, self.variant, self.precision)
        # finalize applies row_scale only where the forward produced it (softmax on tensor cores)
        self._scaled = _lib.prepares_dE_hat(n_local, n_total, M, D, self.variant, self.precision)
        self.peer, self.peer_error = False, None
        world = dist.get_world_size(self.group)
        if peer_memory and world > 1:
            ok = self._scaled and world <= 8 and n_local % 128 == 0 and n_local * world == n_total
            if ok:
                try:
                    self._setup_peer_memory(world, dist.get_rank(self.group))
                except Exception as e:          # no peer mapping on this system: the NCCL path is always there
                    self.peer_error = repr(e)
                    if peer_memory is True:
                        raise
            elif peer_memory is True:
                raise ValueError("peer_memory=True needs the tensor-core softmax path, <= 8 ranks and n_local % 128 == 0")
        if not self.peer:
            self.dC_partial = torch.empty((n_total, D), dtype=f32, device=dev)
            self.dC_local = torch.empty((n_local, D), dtype=f32, device=dev)
        self.red = torch.empty(4, dtype=f32, device=dev)          # {loss, dw, db, -}: zeroed by prep; this rank's partials
        self.dE = torch.empty((n_local, M, D), dtype=f32, device=dev)
        self.grad_out = torch.ones((), dtype=f32, device=dev)
        nbytes = lib().ge2e_b200_workspace_bytes(n_local, n_total, M, D, self.variant, self.precision)
        self._ws = torch.zeros(max(nbytes, 1), dtype=torch.uint8, device=dev)
        self._ws_bytes = nbytes
        # global {loss, dw, db, -} after a step: `red` all-reduced in place (NCCL), or the sum of the ranks' rows
        self.results = self.red_sum if self.peer else self.red
        self.loss, self.dw, self.db = self.results[0], self.results[1], self.results[2]
        self._side = torch.cuda.Stream(device=dev)

    def _setup_peer_memory(self, world: int, rank: int) -> None:
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        f32, dev = torch.float32, self.device
        gname = self.group.group_name
        c_all = symm.empty((self.n_total, self.D), dtype=f32, device=dev)
        hc = symm.rendezvous(c_all, gname)
        dC = symm.empty((self.n_local, self.D), dtype=f32, device=dev)
        hd = symm.rendezvous(dC, gname)
        ptr_c, ptr_d = list(hc.buffer_ptrs), list(hd.buffer_ptrs)
        if len(ptr_c) != world or len(ptr_d) != world:
            raise RuntimeError("symmetric-memory rendezvous returned a different world size")
        off_bytes = self.spk_offset * self.D * 4
        try:
            mc = int(hc.multicast_ptr)
        except Exception:
            mc = 0
        if mc:
            # NVSwitch multicast: one store per element leaves this GPU, the switch writes every rank's copy
            self._peer_slices, self._n_peers, self._mcast = (C.c_void_p * 1)(mc + off_bytes), 1, 1
        else:
            peers = [ptr_c[r] + off_bytes for r in range(world) if r != rank]   # MY slice in every peer's c_hat_all
            self._peer_slices, self._n_peers, self._mcast = (C.c_void_p * len(peers))(*peers), len(peers), 0
        self._dC_owner = (C.c_void_p * world)(*ptr_d)                            # every rank's dC_local, mine included
        self._world = world
        # {loss, dw, db} of every rank: a [world, 4] table replicated on every rank; rank r stores its row into
        # every copy in front of the second barrier, every rank sums the rows itself (no all-reduce kernel)
        red_all = symm.empty((world, 4), dtype=f32, device=dev)
        hr = symm.rendezvous(red_all, gname)
        rows = [p + rank * 16 for p in hr.buffer_ptrs]
        self._red_rows = (C.c_void_p * world)(*rows)
        self.red_all, self._hr = red_all, hr
        self.red_sum = torch.zeros(4, dtype=f32, device=dev)
        self._hc, self._hd = hc, hd
        self.c_hat_all = c_all
        self.c_hat_mine = c_all[self.spk_offset:self.spk_offset + self.n_local]
        self.dC_local, self.dC_partial = dC, None
        self.peer = True

    def _step_peer(self, E_local, w, b) -> None:
        """prep -> publish c_hat slice to the peers, clear my dC rows -> barrier -> step kernel (centroid pass adds
        into the owners' rows over NVLink) -> barrier -> all-reduce {loss, dw, db} || finalize."""
        h, dist = lib(), self.dist
        nl, nt, off, M, D = self.n_local, self.n_total, self.spk_offset, self.M, self.D
        cur = torch.cuda.current_stream(self.device)
        s = cur.cuda_stream
        ws = self._ws.data_ptr() if self._ws_bytes else None
        check(h.ge2e_b200_prep(E_local.data_ptr(), nl, M, D, self.precision, self.e_hat.data_ptr(),
                               self.c_hat_mine.data_ptr(), self.cos_diag.data_ptr(), self.red.data_ptr(), s),
              "ge2e_b200_prep")
        check(h.ge2e_b200_peer_publish(self.c_hat_mine.data_ptr(), self._peer_slices, self._n_peers, self._mcast, nl * D,
                                       self.dC_local.data_ptr(), nl * D, s), "ge2e_b200_peer_publish")
        self._hc.barrier(channel=0)          # every slice of c_hat_all has landed, every dC_local is cleared
        check(h.ge2e_b200_step_rows_peers(self.e_hat.data_ptr(), self.c_hat_all.data_ptr(), self.cos_diag.data_ptr(), nl,
                                          nt, off, M, D, w.data_ptr(), b.data_ptr(), self.eps, self.variant,
                                          self.precision, self.grad_out.data_ptr(), self.row_stat.data_ptr(),
                                          self.row_kstar.data_ptr(), self.row_aux.data_ptr(), self.row_scale.data_ptr(),
                                          self.red.data_ptr(), self.dE_hat.data_ptr(), self._dC_owner, self._world, ws,
                                          self._ws_bytes, s), "ge2e_b200_step_rows_peers")
        check(h.ge2e_b200_peer_publish(self.red.data_ptr(), self._red_rows, self._world, 0, 4, None, 0, s),
              "ge2e_b200_peer_publish")   # my {loss, dw, db} into row `rank` of every rank's table
        self._hd.barrier(channel=0)          # every rank's contributions to my dC rows (and its scalars) have landed
        check(h.ge2e_b200_bwd_finalize(E_local.data_ptr(), self.dE_hat.data_ptr(), self.dC_local.data_ptr(),
                                       self.cos_diag.data_ptr(), self.row_stat.data_ptr(), self.row_aux.data_ptr(),
                                       self.row_scale.data_ptr(), nl, M, D, w.data_ptr(), b.data_ptr(), self.eps,
                                       self.variant, self.grad_out.data_ptr(), self.dE.data_ptr(), s),
              "ge2e_b200_bwd_finalize")
        torch.sum(self.red_all, dim=0, out=self.red_sum)

    def step(self, E_local: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> None:
        if E_local.dtype != torch.float32:
            raise TypeError(f"ShardedGE2EPlan takes float32 embeddings only, got {E_local.dtype}; bfloat16 / float16 "
                            "embeddings run through GE2ELoss(process_group=...) or a single-device GE2EPlan(dtype=...)")
        if self.peer:
            return self._step_peer(E_local, w, b)
        h, dist = lib(), self.dist
        nl, nt, off, M, D = self.n_local, self.n_total, self.spk_offset, self.M, self.D
        s = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._ws.data_ptr() if self._ws_bytes else None
        check(h.ge2e_b200_prep(E_local.data_ptr(), nl, M, D, self.precision, self.e_hat.data_ptr(),
                               self.c_hat_mine.data_ptr(), self.cos_diag.data_ptr(), self.red.data_ptr(), s),
              "ge2e_b200_prep")
        dist.all_gather_into_tensor(self.c_hat_all, self.c_hat_mine, group=self.group)
        s = torch.cuda.current_stream(self.device).cuda_stream
        check(h.ge2e_b200_step_rows(self.e_hat.data_ptr(), self.c_hat_all.data_ptr(), self.cos_diag.data_ptr(), nl, nt,
                                    off, M, D, w.data_ptr(), b.data_ptr(), self.eps, self.variant, self.precision,
                                    self.grad_out.data_ptr(), self.row_stat.data_ptr(), self.row_kstar.data_ptr(),
                                    self.row_aux.data_ptr(), self.row_scale.data_ptr(), self.red.data_ptr(),
                                    self.dE_hat.data_ptr(), self.dC_partial.data_ptr(), ws, self._ws_bytes, s),
              "ge2e_b200_step_rows")
        dist.reduce_scatter_tensor(self.dC_local, self.dC_partial, op=dist.ReduceOp.SUM, group=self.group)
        # {loss, dw, db} are not inputs of finalize: their all-reduce runs beside it (fork / join on a side
        # stream; inside a capture this becomes a parallel branch of the graph)
        cur = torch.cuda.current_stream(self.device)
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            dist.all_reduce(self.red, op=dist.ReduceOp.SUM, group=self.group)
        s = cur.cuda_stream
        check(h.ge2e_b200_bwd_finalize(E_local.data_ptr(), self.dE_hat.data_ptr(), self.dC_local.data_ptr(),
                                       self.cos_diag.data_ptr(), self.row_stat.data_ptr(), self.row_aux.data_ptr(),
                                       self.row_scale.data_ptr() if self._scaled else None, nl,
                                       M, D, w.data_ptr(), b.data_ptr(), self.eps, self.variant,
                                       self.grad_out.data_ptr(), self.dE.data_ptr(), s), "ge2e_b200_bwd_finalize")
        cur.wait_stream(self._side)

    def capture(self, E_local, w: torch.Tensor, b: torch.Tensor, steps: int = 1):
        """``steps`` consecutive sharded steps in one CUDA graph (NCCL collectives included).
        ``E_local`` is one batch or a list of batches the steps rotate over."""
        batches = list(E_local) if isinstance(E_local, (list, tuple)) else [E_local]
        with torch.cuda.device(self.device):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    self.step(batches[0], w, b)          # warm-up: communicator set-up, lazy attributes
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for k in range(steps):
                    self.step(batches[k % len(batches)], w, b)
        return g


class _HostFeed:
    """Slot machinery shared by the host-fed plans: ``depth`` device buffers, one CUDA graph per slot
    holding that slot's whole step plus the device->host read of its result, a copy stream for the
    H2D transfers and a compute stream for the graphs."""

    def _setup(self, shape, depth, device, make_plan, result_of):
        self.device = torch.device(device if device is not None else "cuda")
        self.shape, self.depth = tuple(shape), depth
        dev = self.device
        self.plans = [make_plan() for _ in range(depth)]
        self.bufs = [torch.empty(self.shape, dtype=torch.float32, device=dev) for _ in range(depth)]
        self.results = [torch.zeros(3, dtype=torch.float32).pin_memory() for _ in range(depth)]
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.compute_stream = torch.cuda.Stream(device=dev)
        self._copied = [torch.cuda.Event() for _ in range(depth)]
        self._done = [torch.cuda.Event() for _ in range(depth)]
        self._used = [False] * depth
        self._k = 0
        self._graphs = []
        with torch.cuda.device(dev):
            for i in range(depth):
                p, buf, res = self.plans[i], self.bufs[i], self.results[i]
                buf.normal_()
                torch.cuda.synchronize()
                with torch.cuda.stream(self.compute_stream):
                    for _ in range(2):
                        p.step(buf, self.w, self.b)         # warm-up outside capture (communicators, lazy attributes)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                before = lib().ge2e_b200_launch_count()
                with torch.cuda.graph(g, stream=self.compute_stream):
                    p.step(buf, self.w, self.b)
                    for dst, src in result_of(p, res):
                        dst.copy_(src, non_blocking=True)
                self.launches_per_step = lib().ge2e_b200_launch_count() - before
                self._graphs.append(g)

    def submit(self, E_host: torch.Tensor) -> int:
        n = 1
        for d in self.shape:
            n *= d
        if not (E_host.dtype == torch.float32 and E_host.is_contiguous() and E_host.numel() == n):
            raise ValueError(f"submit: expected a contiguous fp32 batch of {n} values (the host-fed plans take float32 "
                             f"embeddings only, got {E_host.dtype})")
        if E_host.device.type == "cpu" and not E_host.is_pinned():
            raise ValueError("submit: the host batch must be in pinned memory (an unpinned copy is synchronous)")
        i = self._k % self.depth
        self._k += 1
        cs, ms = self.copy_stream, self.compute_stream
        if self._used[i]:
            cs.wait_event(self._done[i])                 # slot's previous step has consumed its buffer
        with torch.cuda.stream(cs):
            self.bufs[i].copy_(E_host.view(self.shape), non_blocking=True)
            self._copied[i].record(cs)
        ms.wait_event(self._copied[i])
        with torch.cuda.stream(ms):
            self._graphs[i].replay()
            self._done[i].record(ms)
        self._used[i] = True
        return i

    def result(self, ticket: int):
        """(loss, dw, db) of the slot as Python floats; blocks until that slot's step has finished."""
        self._done[ticket].synchronize()
        r = self.results[ticket]
        return float(r[0]), float(r[1]), float(r[2])

    def dE(self, ticket: int) -> torch.Tensor:
        """Device gradient of the slot's batch (valid for work queued after ``done_event(ticket)``)."""
        return self.plans[ticket].dE

    def done_event(self, ticket: int) -> torch.cuda.Event:
        return self._done[ticket]


class GE2EHostFeed(_HostFeed):
    """fwd+bwd over HOST-resident batches, pipelined: the H2D copy of batch k+1 (copy stream) runs
    under the fwd+bwd of batch k (compute stream), and every slot's step -- the four stages plus the
    device->host read of {loss, dw, db} into the slot's pinned result -- is one CUDA graph, so a
    ``submit`` costs a handful of stream calls on the host.  This is the trainer's call sequence
    (s4_train_embed_model.py:170-200: batch from the loader -> ``.to(device)`` -> loss -> backward ->
    ``loss.to("cpu")``) with the loader's pinned batch as the input.

        feed = GE2EHostFeed(N, M, D, w, b, precision="tf32")
        t = feed.submit(E_pinned)          # returns at once
        loss, dw, db = feed.result(t)      # waits for that slot; dE of the slot: feed.dE(t) (device)

    ``depth`` slots are in flight at most; ``submit`` on a slot still in use waits on the device
    (stream order), never on the host.  ``w`` / ``b`` are read at replay time, so in-place optimiser
    updates between submits are seen."""

    def __init__(self, N: int, M: int, D: int, w: torch.Tensor, b: torch.Tensor, variant: str = "softmax",
                 precision: str = "fp32", eps: float = 1e-6, device=None, depth: int = 2):
        self.N, self.M, self.D = N, M, D
        self.w, self.b = w, b
        dev = torch.device(device if device is not None else "cuda")
        self._setup((N, M, D), depth, dev, lambda: GE2EPlan(N, M, D, variant, precision, eps, device=dev),
                    lambda p, res: [(res, p._accum[0:3])])
        self.path = self.plans[0].path


class ShardedGE2EHostFeed(_HostFeed):
    """``GE2EHostFeed`` for the speaker-sharded step (one process per GPU): every rank submits ITS shard
    [n_local, M, D] from pinned host memory; a slot's graph holds the four stages, the three NCCL
    collectives and the read-back of the global {loss, dw, db}.  Both slots' graphs run on the one
    compute stream, so the communicator sees its collectives in the same order on every rank as long as
    all ranks submit in lockstep (same number of submits, as a data-parallel loop does)."""

    def __init__(self, n_local: int, n_total: int, spk_offset: int, M: int, D: int, w: torch.Tensor, b: torch.Tensor,
                 variant: str = "softmax", precision: str = "tf32", eps: float = 1e-6, group=None, device=None,
                 depth: int = 2):
        self.w, self.b = w, b
        dev = torch.device(device if device is not None else "cuda")
        self._setup((n_local, M, D), depth, dev,
                    lambda: ShardedGE2EPlan(n_local, n_total, spk_offset, M, D, variant, precision, eps, group, dev),
                    lambda p, res: [(res, p.results[0:3])])
