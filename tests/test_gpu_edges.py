"""GPU tests at the edges the well-behaved parity inputs never reach, every kernel family against the float64
oracles (oracle/ge2e_oracle.py for small shapes, oracle/ge2e_oracle_torch.py on the device for N >= 129):

  * degenerate batches: a zero utterance row, a zero centroid, a zero leave-one-out centroid, rows and a
    centroid whose norm sits just below / above the cosine clamp delta = 1e-8, a collapsed speaker and a
    duplicated speaker -- F.cosine_similarity's gradient below the clamp (value clamped, derivative x / |x|
    kept) on the single-kernel step, the SIMT pipeline, TF32, split-fp16, f16, hybrid and speaker shards;
  * contiguous inputs at a storage offset of 1, 2 or 3 floats (E not 16-byte aligned);
  * exact ties in the contrast arg-max (the header promises the lowest k);
  * both sides of every shape selector, and the backward's shared-memory envelope;
  * large w (logits far below the tensor-core path's fixed shift |w| + b).

Each case asserts which path ran (ge2e_b200_path, plan.path, plan.single_kernel) so that a dispatch change cannot
make it test something else.  Tolerances as in test_gpu_parity.py: fp32 1e-5, TF32 / f16 2e-3, db absolute 1e-5 U.
"""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_oracle_torch as orct

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
TF32_TOL = 2e-3
TOL = {"fp32": FP32_TOL, "fp32_simt": FP32_TOL, "fp32_split": FP32_TOL, "tf32": TF32_TOL, "f16": TF32_TOL}
DEV = "cuda:0"
DELTA = orc.COS_DELTA
EPS = 1e-6


@pytest.fixture(scope="module")
def pkg():
    import speaker_embedding_ge2e_loss_b200 as p
    p.lib()  # fails loudly when the CUDA library is missing
    assert torch.cuda.is_available()
    return p


class small_step_mode:
    """ge2e_b200_debug_small_step for the duration of a block (1 = the default rule)."""

    def __init__(self, pkg, mode):
        self.h, self.mode = pkg.lib(), mode

    def __enter__(self):
        self.h.ge2e_b200_debug_small_step(self.mode)

    def __exit__(self, *a):
        self.h.ge2e_b200_debug_small_step(1)


# ------------------------------------------------------------------ helpers
def codes(pkg, N, M, D, precision, variant):
    from speaker_embedding_ge2e_loss_b200 import _lib
    v = _lib.VARIANTS[variant]
    return v, _lib.resolve_precision(precision, N, N, M, D, v)


def reference(E_np, w, b, variant, g=1.0):
    """float64 truth: the numpy oracle for small batches, the torch restatement on the device for large ones."""
    N, M, D = E_np.shape
    if N * M * D <= 300_000:
        r = orc.forward_backward(E_np, w, b, EPS, variant, g=g)
        r["dE"] = torch.tensor(r["dE"], device=DEV)
        return r
    return orct.forward_backward(torch.tensor(E_np, device=DEV), w, b, EPS, variant, g=g)


def trel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def check(got, ref, U, tol, degenerate=()):
    """loss, dw, db; dE separately on the degenerate speakers and on all other rows (a zero row's gradient is
    ~1/delta and would hide an error on the normal rows)."""
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), (got["loss"], ref["loss"])
    dE, rE = got["dE"].reshape(ref["dE"].shape), ref["dE"]
    N = rE.shape[0]
    deg = torch.zeros(N, dtype=torch.bool, device=rE.device)
    deg[list(degenerate)] = True
    assert torch.isfinite(dE).all()
    for part in (deg, ~deg):
        if part.any():
            r = trel(dE[part], rE[part])
            assert r <= tol, (r, "degenerate" if part is deg else "normal")
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"])), (got["dw"], ref["dw"])
    assert abs(got["db"] - ref["db"]) <= 1e-5 * U, (got["db"], ref["db"])


def run_module(pkg, E, w, b, precision, variant, g=1.0):
    crit = pkg.GE2ELoss(None, device=E.device, w=w, b=b, variant=variant, precision=precision)
    Eg = E.detach().requires_grad_(True)
    loss = crit(Eg)
    (loss * g).backward()
    torch.cuda.synchronize()
    return dict(loss=loss.item(), dE=Eg.grad.clone(), dw=crit.w.grad.item(), db=crit.b.grad.item())


def run_unperm(pkg, E, w, b, precision, variant, seed=0):
    """The module with unperm=: E handed over as [U, D] in a shuffled row order."""
    N, M, D = E.shape
    U = N * M
    perm = torch.randperm(U, generator=torch.Generator().manual_seed(seed)).to(E.device)
    unperm = torch.empty_like(perm)
    unperm[perm] = torch.arange(U, device=E.device)
    shuffled = E.reshape(U, D)[perm].contiguous()
    crit = pkg.GE2ELoss(None, device=E.device, w=w, b=b, variant=variant, precision=precision)
    Eg = shuffled.requires_grad_(True)
    loss = crit(Eg, unperm=unperm, speakers=N)
    loss.backward()
    torch.cuda.synchronize()
    return dict(loss=loss.item(), dE=Eg.grad[unperm].reshape(N, M, D), dw=crit.w.grad.item(), db=crit.b.grad.item())


def run_plan(pkg, E, w, b, precision, variant):
    N, M, D = E.shape
    plan = pkg.GE2EPlan(N, M, D, variant, precision, device=E.device)
    wt, bt = torch.tensor(float(w), device=E.device), torch.tensor(float(b), device=E.device)
    plan.step(E, wt, bt)
    torch.cuda.synchronize()
    return dict(loss=plan.loss.item(), dE=plan.dE.clone(), dw=plan.dw.item(), db=plan.db.item(),
                kstar=plan.row_kstar.clone()), plan


def run_shards(pkg, E, w, b, R, precision, variant=0):
    """R speaker shards on one GPU through the staged C-ABI calls (as in test_gpu_step.py): prep per shard into
    a shared c_hat_all (the all-gather), forward / backward rows with spk_offset, the full-height dC_hat partials
    summed here (the reduce-scatter), finalize per shard."""
    from speaker_embedding_ge2e_loss_b200 import ops, _lib
    N, M, D = E.shape
    nl = N // R
    prec = _lib.PRECISIONS[precision]
    dev = E.device
    wt, bt = torch.tensor(float(w), device=dev), torch.tensor(float(b), device=dev)
    gone = torch.ones((), device=dev)
    c_hat_all = torch.empty((N, D), device=dev)
    st = []
    for r in range(R):
        Er = E[r * nl:(r + 1) * nl].contiguous()
        e_hat, cos_diag, accum = ops.prep(Er, c_hat_all[r * nl:(r + 1) * nl], prec)
        st.append(dict(E=Er, e_hat=e_hat, cos_diag=cos_diag, accum=accum))
    dC_sum = torch.zeros((N, D), dtype=torch.float64, device=dev)
    loss = dw = db = 0.0
    for r, s in enumerate(st):
        rs, ks, aux, _, _, dE_hat, row_scale = ops.fwd_rows(s["e_hat"], c_hat_all, s["cos_diag"], nl, N, r * nl, M, D,
                                                            wt, bt, EPS, variant, prec, s["accum"], want_grad=True)
        s["dE_hat"], dC_part, dwdb = ops.bwd_rows(s["e_hat"], c_hat_all, s["cos_diag"], rs, ks, aux, nl, N, r * nl, M, D,
                                                  wt, bt, EPS, variant, prec, gone, dE_hat=dE_hat, row_scale=row_scale)
        s["row_stat"], s["row_aux"], s["row_scale"] = rs, aux, row_scale
        torch.cuda.synchronize()
        dC_sum += dC_part.double()
        loss += s["accum"][0].item()
        dw += dwdb[0].item()
        db += dwdb[1].item()
    dE = []
    for r, s in enumerate(st):
        dC_local = dC_sum[r * nl:(r + 1) * nl].float().contiguous()
        dE.append(ops.bwd_finalize(s["E"], s["dE_hat"], dC_local, s["cos_diag"], s["row_stat"], s["row_aux"], wt, bt,
                                   EPS, variant, gone, row_scale=s["row_scale"]))
    torch.cuda.synchronize()
    return dict(loss=loss, dE=torch.cat(dE, dim=0), dw=dw, db=db)


# ------------------------------------------------------------------ degenerate batches
DEGENERATE = list(range(1, 12))


def degenerate_batch(N, M, D, seed=0):
    """A clustered batch with speakers 1..11 degenerate, built so that every sum the kernels form is exact in
    fp32 (cancelling pairs next to zero rows; a + (-a + t) with |a| >> |t| is exact by Sterbenz's lemma):
      1 zero utterance row            2 zero centroid (e, -e, zeros)
      3 zero leave-one-out centroid of the last row (e, -e, zeros, f)
      4..7 one row of norm 0.5, 0.999, 1.001, 2 delta
      8 centroid of norm 0.5 delta (a, -a + t, zeros)
      9 collapsed speaker (all rows equal)    10, 11 bit-identical speakers"""
    assert N >= 12 and M >= 3
    E = orc.make_embeddings(N, M, D, seed=seed, kind="clustered")
    rng = np.random.default_rng(seed + 1)

    def unit():
        v = rng.standard_normal(D)
        return v / np.linalg.norm(v)

    E[1, 1] = 0.0
    p = E[2, 0].copy()
    E[2] = 0.0
    E[2, 0], E[2, 1] = p, -p
    f = E[3, M - 1].copy()
    E[3] = 0.0
    E[3, 0], E[3, 1], E[3, M - 1] = p, -p, f
    for j, s in zip((4, 5, 6, 7), (0.5, 0.999, 1.001, 2.0)):
        E[j, 0] = (E[j, 0].astype(np.float64) * (s * DELTA / np.linalg.norm(E[j, 0].astype(np.float64)))).astype(np.float32)
    a = (1e-6 * unit()).astype(np.float32)
    bvec = (-a.astype(np.float64) + 0.5 * DELTA * M * unit()).astype(np.float32)
    E[8] = 0.0
    E[8, 0], E[8, 1] = a, bvec
    E[9] = E[9, 0]
    E[11] = E[10]
    return E


# family: (N, M, D, precision, small-step mode, expected ge2e_b200_path, expected single_kernel, variants)
FAMILIES = {
    "small_step_fast_d256": (16, 4, 256, "fp32", 1, 0, True, ("softmax", "contrast")),
    "small_step_slow_d100": (16, 5, 100, "fp32", 1, 0, True, ("softmax", "contrast")),
    "simt_pipeline_m20": (16, 20, 256, "fp32", 0, 0, False, ("softmax", "contrast")),
    "simt_pipeline_m40": (16, 40, 256, "fp32", 0, 0, False, ("softmax", "contrast")),
    "tf32_d128": (300, 4, 128, "tf32", 1, 1, False, ("softmax",)),
    "tf32_d160": (300, 4, 160, "tf32", 1, 1, False, ("softmax",)),
    "split_d256": (300, 4, 256, "fp32", 1, 2, False, ("softmax",)),
    "f16_d256": (300, 4, 256, "f16", 1, 3, False, ("softmax",)),
}


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_degenerate_rows_every_family(pkg, family):
    N, M, D, precision, mode, path, single, variants = FAMILIES[family]
    tol = TOL[precision]
    E_np = degenerate_batch(N, M, D, seed=N + M + D)
    E = torch.tensor(E_np, device=DEV)
    with small_step_mode(pkg, mode):
        for variant in variants:
            vcode, pcode = codes(pkg, N, M, D, precision, variant)
            assert pkg.lib().ge2e_b200_path(N, N, M, D, vcode, pcode) == path
            ref = reference(E_np, 10.0, -5.0, variant)
            got, plan = run_plan(pkg, E, 10.0, -5.0, precision, variant)
            assert plan.path == path and plan.single_kernel == single
            check(got, ref, N * M, tol, DEGENERATE)
            check(run_module(pkg, E, 10.0, -5.0, precision, variant), ref, N * M, tol, DEGENERATE)
            check(run_unperm(pkg, E, 10.0, -5.0, precision, variant), ref, N * M, tol, DEGENERATE)
            if variant == "softmax":        # upstream gradient != 1 scales the cached step's gradients
                check(run_module(pkg, E, 10.0, -5.0, precision, variant, g=-0.7),
                      reference(E_np, 10.0, -5.0, variant, g=-0.7), N * M, tol, DEGENERATE)


def test_degenerate_rows_hybrid_operand_copies(pkg):
    # a shape no other test has run: the module caches its workspace size per shape, queried with the mode set
    N, M, D = 300, 5, 128
    E_np = degenerate_batch(N, M, D, seed=9)
    E = torch.tensor(E_np, device=DEV)
    ref = reference(E_np, 10.0, -5.0, "softmax")
    h = pkg.lib()
    h.ge2e_b200_debug_hybrid(1)
    try:
        got, plan = run_plan(pkg, E, 10.0, -5.0, "tf32", "softmax")
        assert plan.path == 1
        mod = run_module(pkg, E, 10.0, -5.0, "tf32", "softmax")
    finally:
        h.ge2e_b200_debug_hybrid(0)
    check(got, ref, N * M, TF32_TOL, DEGENERATE)
    check(mod, ref, N * M, TF32_TOL, DEGENERATE)


@pytest.mark.parametrize("N,M,D,precision,variant", [
    (48, 4, 256, "fp32", "softmax"), (48, 4, 256, "fp32", "contrast"), (384, 4, 128, "tf32", "softmax"),
])
def test_degenerate_rows_three_speaker_shards(pkg, N, M, D, precision, variant):
    from speaker_embedding_ge2e_loss_b200 import _lib
    E_np = degenerate_batch(N, M, D, seed=3)
    E = torch.tensor(E_np, device=DEV)
    if precision == "tf32":
        assert pkg.lib().ge2e_b200_path(N // 3, N, M, D, 0, _lib.TF32) == 1
    ref = reference(E_np, 10.0, -5.0, variant)
    got = run_shards(pkg, E, 10.0, -5.0, 3, precision, _lib.VARIANTS[variant])
    check(got, ref, N * M, TOL[precision], DEGENERATE)


def test_single_speaker_batch(pkg):
    """N = 1: no negatives; the loss is eps-driven (dE ~ 1e-6, fp32 rounding of S gives ~1e-4 relative, as the
    golden one-speaker case in test_gpu_parity.py)."""
    E_np = orc.make_embeddings(1, 5, 256, seed=1, kind="clustered")
    E = torch.tensor(E_np, device=DEV)
    for variant in ("softmax", "contrast"):
        ref = reference(E_np, 10.0, -5.0, variant)
        got, plan = run_plan(pkg, E, 10.0, -5.0, "fp32", variant)
        assert plan.single_kernel
        assert abs(got["loss"] - ref["loss"]) <= FP32_TOL * max(1.0, abs(ref["loss"]))
        assert trel(got["dE"], ref["dE"]) <= 2e-4
        if variant == "contrast":
            assert (got["kstar"][:5] == -1).all()


# ------------------------------------------------------------------ unaligned inputs
def at_offset(E, off):
    """E's values in a contiguous tensor that starts `off` floats into its allocation."""
    buf = torch.zeros(off + E.numel() + 4, dtype=torch.float32, device=E.device)
    out = buf[off:off + E.numel()].view(E.shape)
    out.copy_(E)
    assert out.is_contiguous() and (out.data_ptr() % 16 == 0) == (off % 4 == 0)
    return out


UNALIGNED = {     # (N, M, D, precision, small-step mode, path, variants)
    "small_step": (16, 4, 256, "fp32", 1, 0, ("softmax", "contrast")),
    "simt_pipeline": (16, 20, 256, "fp32", 0, 0, ("softmax", "contrast")),
    "tf32": (300, 4, 128, "tf32", 1, 1, ("softmax",)),      # contrast on TF32: near-tied arg-maxes may flip
    "split": (300, 4, 256, "fp32", 1, 2, ("softmax",)),
    "f16": (300, 4, 256, "f16", 1, 3, ("softmax",)),
}


@pytest.mark.parametrize("off", [0, 1, 2, 3])
@pytest.mark.parametrize("family", sorted(UNALIGNED))
def test_unaligned_input(pkg, family, off):
    from speaker_embedding_ge2e_loss_b200 import ops
    N, M, D, precision, mode, path, variants = UNALIGNED[family]
    tol = TOL[precision]
    E_np = orc.make_embeddings(N, M, D, seed=off + 40, kind="raw")
    E0 = torch.tensor(E_np, device=DEV)
    E = at_offset(E0, off)
    with small_step_mode(pkg, mode):
        for variant in variants:
            vcode, pcode = codes(pkg, N, M, D, precision, variant)
            assert pkg.lib().ge2e_b200_path(N, N, M, D, vcode, pcode) == path
            ref = reference(E_np, 10.0, -5.0, variant)
            aligned = run_module(pkg, E0, 10.0, -5.0, precision, variant)
            got = run_module(pkg, E, 10.0, -5.0, precision, variant)
            check(got, ref, N * M, tol)
            assert abs(got["loss"] - aligned["loss"]) <= 1e-5 * abs(aligned["loss"])
            assert trel(got["dE"], aligned["dE"]) <= tol
            # the speaker-major input handed over as [U, D] rows at the same offset, with unperm
            U = N * M
            Eu = at_offset(E0.reshape(U, D), off)
            crit = pkg.GE2ELoss(None, device=E.device, w=10.0, b=-5.0, variant=variant, precision=precision)
            Eg = Eu.requires_grad_(True)
            loss = crit(Eg, unperm=torch.arange(U, device=DEV), speakers=N)
            loss.backward()
            check(dict(loss=loss.item(), dE=Eg.grad.reshape(N, M, D), dw=crit.w.grad.item(), db=crit.b.grad.item()),
                  ref, U, tol)
            # the custom op (what torch.compile sees)
            w, b = torch.tensor(10.0, device=DEV, requires_grad=True), torch.tensor(-5.0, device=DEV, requires_grad=True)
            Eg = at_offset(E0, off).requires_grad_(True)
            lo = ops.ge2e_fwd(Eg, w, b, EPS, vcode, pcode)[0]
            lo.backward()
            check(dict(loss=lo.item(), dE=Eg.grad, dw=w.grad.item(), db=b.grad.item()), ref, U, tol)
            # a plan copies nothing behind the caller's back: the fp16-plane precisions refuse such an E
            if pcode in (2, 3) and off % 4:
                with pytest.raises(ValueError, match="16-byte"):
                    run_plan(pkg, E, 10.0, -5.0, precision, variant)
            else:
                got, plan = run_plan(pkg, E, 10.0, -5.0, precision, variant)
                assert plan.path == path
                check(got, ref, U, tol)


# ------------------------------------------------------------------ exact contrast ties
def one_hot_batch(N, M, D, dup, seed=0):
    """Every utterance row is one +1 entry, so every e . c_hat is one entry of c_hat -- no rounding in the
    sum, TF32 included -- and all centroid entries are count / sqrt(sum count^2) with counts of M = 4 rows: far
    apart unless equal.  Speakers of `dup` are bit-identical copies of the first one: exact ties."""
    rng = np.random.default_rng(seed)
    E = np.zeros((N, M, D), dtype=np.float32)
    dims = rng.integers(0, D, size=(N, M))
    for j in range(N):
        for i in range(M):
            E[j, i, dims[j, i]] = 1.0
    for a, b in dup:
        E[b] = E[a]
    return E


@pytest.mark.parametrize("family", ["simt_pipeline", "small_step", "tf32"])
def test_contrast_exact_ties_take_the_lowest_k(pkg, family):
    from speaker_embedding_ge2e_loss_b200 import ops
    M, D = 4, 128
    if family == "small_step":
        N, dup, mode, precision = 128, [(5, 100), (7, 9)], 1, "fp32"
    else:
        N, dup, mode, precision = 300, [(5, 260), (7, 9)], 0, ("tf32" if family == "tf32" else "fp32")
    E_np = one_hot_batch(N, M, D, dup, seed=N)
    ref = orc.forward_backward(E_np, 10.0, -5.0, EPS, "contrast")
    kref = torch.tensor(ref["kstar"].reshape(-1), device=DEV, dtype=torch.int32)
    E = torch.tensor(E_np, device=DEV)
    vcode, pcode = codes(pkg, N, M, D, precision, "contrast")
    with small_step_mode(pkg, mode):
        got, plan = run_plan(pkg, E, 10.0, -5.0, precision, "contrast")
        assert plan.single_kernel == (family == "small_step")
        assert plan.path == (1 if family == "tf32" else 0)
        assert torch.equal(got["kstar"], kref)
        check(got, dict(ref, dE=torch.tensor(ref["dE"], device=DEV)), N * M, TOL[precision])
        # the forward rows kernel alone, through ge2e_b200_fwd_rows
        c_hat = torch.empty((N, D), device=DEV)
        e_hat, cos_diag, accum = ops.prep(E, c_hat, pcode)
        wt, bt = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
        _, kstar, _, _, _, _, _ = ops.fwd_rows(e_hat, c_hat, cos_diag, N, N, 0, M, D, wt, bt, EPS, vcode, pcode, accum)
        torch.cuda.synchronize()
        assert torch.equal(kstar, kref)
    # the fixture does produce what it is about: many rows have a tied hardest negative, some of them the copies
    Eh = E.reshape(N * M, D).double()
    Ch = torch.nn.functional.normalize(E.double().mean(1), dim=1)
    S = Eh @ Ch.T
    rows = torch.arange(N * M, device=DEV)
    S[rows, rows // M] = -float("inf")
    n_max = (S == S.max(dim=1, keepdim=True).values).sum(dim=1)
    assert (n_max > 1).float().mean().item() > 0.1
    spk = rows // M
    for a, b in dup:
        assert (kref[spk != a] == a).any().item()
        assert not (kref[spk != a] == b).any().item()     # outside speaker a, a copy never wins over its original


# ------------------------------------------------------------------ shape selectors and the backward's envelope
def run_and_check(pkg, N, M, D, precision="fp32", mode=0, variant="softmax", kind="clustered"):
    E_np = orc.make_embeddings(N, M, D, seed=N + M + D, kind=kind)
    E = torch.tensor(E_np, device=DEV)
    ref = reference(E_np, 10.0, -5.0, variant)
    with small_step_mode(pkg, mode):
        got, plan = run_plan(pkg, E, 10.0, -5.0, precision, variant)
    check(got, ref, N * M, TF32_TOL if plan.path in (1, 3) else FP32_TOL)
    return plan


@pytest.mark.parametrize("M", [4, 5, 8, 9, 12, 13, 16, 17])
def test_register_row_buckets(pkg, M):
    """prep_reg / finalize_reg instantiate 4 / 8 / 12 / 16 rows; M = 17 leaves them for the streaming kernels."""
    for variant in ("softmax", "contrast"):
        plan = run_and_check(pkg, 8, M, 256, variant=variant)
        assert plan.path == 0 and not plan.single_kernel


@pytest.mark.parametrize("D", [128, 256, 512])
@pytest.mark.parametrize("M", [32, 33])
def test_warp_kernel_row_limit(pkg, M, D):
    """finalize's warp-per-speaker kernel takes M <= 32; M = 33 goes to the shared-memory kernel."""
    plan = run_and_check(pkg, 6, M, D, kind="raw")
    assert plan.path == 0


@pytest.mark.parametrize("D", [127, 128, 129, 255, 257, 511, 513, 1023, 1024])
def test_strip_width_buckets(pkg, D):
    plan = run_and_check(pkg, 8, 4, D, kind="raw")
    assert plan.path == 0


@pytest.mark.parametrize("D", [160, 224])
def test_tf32_slab_counts(pkg, D):
    plan = run_and_check(pkg, 300, 3, D, precision="tf32")
    assert plan.path == 1


@pytest.mark.parametrize("N", [128, 129])
def test_tensor_core_entry(pkg, N):
    plan = run_and_check(pkg, N, 2, 128, precision="tf32", mode=1)
    assert plan.path == (1 if N == 129 else 0)


# (D, largest M whose backward runs): the last stage keeps 2 M + 2 rows in 200 KB of shared memory
ENVELOPE = [(256, 99), (512, 49), (768, 32), (1024, 24), (1000, 24)]


@pytest.mark.parametrize("D,M_max", ENVELOPE)
def test_backward_envelope_both_sides(pkg, D, M_max):
    h = pkg.lib()
    assert h.ge2e_b200_max_utterances(D) == M_max
    run_and_check(pkg, 4, M_max, D, kind="raw")                 # inside: computed, against the oracle
    M = M_max + 1                                               # outside: refused before anything is launched
    E = torch.tensor(orc.make_embeddings(4, M, D, seed=M, kind="raw"), device=DEV)
    crit = pkg.GE2ELoss(None, device=DEV)
    with pytest.raises(ValueError, match="utterances per speaker"):
        crit(E.clone().requires_grad_(True))
    plan = pkg.GE2EPlan(4, M, D, "softmax", "fp32", device=DEV)
    w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
    with pytest.raises(ValueError, match="utterances per speaker"):
        plan.step(E, w, b)
    before = h.ge2e_b200_launch_count()
    rc = h.ge2e_b200_forward_backward(E.data_ptr(), None, 4, M, D, w.data_ptr(), b.data_ptr(), EPS, 0, plan.precision,
                                      plan.grad_out.data_ptr(), plan.e_hat.data_ptr(), plan.c_hat.data_ptr(),
                                      plan.cos_diag.data_ptr(), plan.row_stat.data_ptr(), plan.row_kstar.data_ptr(),
                                      plan.row_aux.data_ptr(), plan.row_scale.data_ptr(), plan._accum.data_ptr(),
                                      plan.dE_hat.data_ptr(), plan.dC_hat.data_ptr(), plan.dE.data_ptr(), None, 0,
                                      torch.cuda.current_stream().cuda_stream)
    assert rc == -2 and h.ge2e_b200_launch_count() == before
    if D in (256, 512):     # aligned rows of a warp-kernel width: the forward alone still runs such a shape
        plan.step(E, w, b, backward=False)
        ref = orc.forward(E.cpu().numpy(), 10.0, -5.0, EPS, "softmax")[0]
        assert abs(plan.loss.item() - ref) <= FP32_TOL * abs(ref)


def test_backward_envelope_on_the_tensor_core_path(pkg):
    """finalize is shared: the tensor-core path has the same envelope (D = 256: 99 utterances)."""
    h = pkg.lib()
    assert h.ge2e_b200_path(129, 129, 99, 256, 0, 1) == 1
    run_and_check(pkg, 129, 99, 256, precision="tf32")
    E = torch.tensor(orc.make_embeddings(129, 100, 256, seed=5, kind="clustered"), device=DEV)
    for precision in ("tf32", "fp32"):
        with pytest.raises(ValueError, match="utterances per speaker"):
            pkg.GE2ELoss(None, device=DEV, precision=precision)(E.clone().requires_grad_(True))
    with pytest.raises(ValueError, match="utterances per speaker"):     # unaligned: the same limit
        pkg.GE2ELoss(None, device=DEV)(at_offset(E[:4], 1).requires_grad_(True))


# ------------------------------------------------------------------ large w, logits far below the fixed shift
def antipodal_batch(N, M, D, seed):
    """Clustered batch whose utterance (0, 0) points away from its speaker: every logit of its row is far below
    |w| + b, its own one by 2 |w|."""
    E = orc.make_embeddings(N, M, D, seed=seed, kind="clustered")
    c = E[0, 1:].sum(0)
    E[0, 0] = -c / np.linalg.norm(c)
    return E


@pytest.mark.parametrize("w", [44.0, 60.0, 80.0])
@pytest.mark.parametrize("precision,N,D,path", [
    ("tf32", 300, 128, 1), ("fp32_split", 300, 256, 2), ("fp32_simt", 64, 256, 0),
])
def test_large_w(pkg, w, precision, N, D, path):
    b = -5.0
    assert w + b < 88                  # the reference's un-stabilised exp(S) stays finite
    M = 4
    E_np = antipodal_batch(N, M, D, seed=int(w))
    E = torch.tensor(E_np, device=DEV)
    ref = reference(E_np, w, b, "softmax")
    got, plan = run_plan(pkg, E, w, b, precision, "softmax")
    assert plan.path == path
    check(got, ref, N * M, TOL[precision])
    check(run_module(pkg, E, w, b, precision, "softmax"), ref, N * M, TOL[precision])
