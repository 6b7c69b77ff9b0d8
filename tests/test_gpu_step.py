"""GPU parity tests of the tensor-core STEP kernel (rows pass + centroid pass, one launch or two) and of
the sharded entry points with spk_offset > 0 / n_local < n_total, against the float64 oracles.

  * full BASELINE sizes (config 3 and config 4) against ``oracle/ge2e_oracle_torch.py`` evaluated in float64
    on the device (itself checked against the numpy oracle here at config 2);
  * R speaker shards emulated on ONE GPU: every shard runs the C-ABI stages with its own spk_offset, the
    full-height dC_hat partials are summed on the host side of the test (what the reduce-scatter does),
    and loss / dE / dw / db must equal the single-batch oracle -- for the fp32 kernels and for the
    tensor-core kernels, through the two-launch path (forward rows, backward rows) and the one-launch path
    (``ge2e_b200_step_rows``);
  * the contrast loss on the tensor-core forward: dE on the rows whose arg-max is robust to TF32 rounding.

Tolerances as in test_gpu_parity.py (BASELINE.json north_star): fp32 1e-5, TF32 2e-3, db absolute.
"""
import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_oracle_torch as orct

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
TF32_TOL = 2e-3
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    import speaker_embedding_ge2e_loss_b200 as p
    p.lib()  # fails loudly when the CUDA library is missing
    assert torch.cuda.is_available()
    return p


def trel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def check_dev(got, ref, U, tol):
    """got / ref: dict(loss, dE (device tensor), dw, db)."""
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), (got["loss"], ref["loss"])
    r = trel(got["dE"].reshape(-1), ref["dE"].reshape(-1))
    assert r <= tol, r
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"])), (got["dw"], ref["dw"])
    assert abs(got["db"] - ref["db"]) <= 1e-5 * U, (got["db"], ref["db"])


def run_plan(pkg, E, w, b, precision, variant="softmax"):
    N, M, D = E.shape
    plan = pkg.GE2EPlan(N, M, D, variant, precision, device=E.device)
    wt = torch.tensor(float(w), device=E.device)
    bt = torch.tensor(float(b), device=E.device)
    plan.step(E, wt, bt)
    torch.cuda.synchronize()
    return dict(loss=plan.loss.item(), dE=plan.dE.clone(), dw=plan.dw.item(), db=plan.db.item()), plan


def run_module(pkg, E, w, b, precision, variant="softmax", g=None):
    crit = pkg.GE2ELoss(None, device=E.device, w=w, b=b, variant=variant, precision=precision)
    Eg = E.clone().requires_grad_(True)
    loss = crit(Eg)
    (loss if g is None else loss * g).backward()
    torch.cuda.synchronize()
    return dict(loss=loss.item(), dE=Eg.grad, dw=crit.w.grad.item(), db=crit.b.grad.item())


# ------------------------------------------------------------------ the checker itself, on the device
@pytest.mark.parametrize("variant", ["softmax", "contrast"])
def test_torch_oracle_on_device_matches_numpy_oracle(variant):
    N, M, D = 64, 10, 256                                                     # BASELINE config 2
    E = orc.make_embeddings(N, M, D, seed=2, kind="clustered")
    ref = orc.forward_backward(E, 10.0, -5.0, 1e-6, variant, g=0.5)
    got = orct.forward_backward(torch.tensor(E, device=DEV), 10.0, -5.0, 1e-6, variant, g=0.5, chunk=100)
    assert abs(got["loss"] - ref["loss"]) <= 1e-11 * abs(ref["loss"])
    assert np.linalg.norm(got["dE"].cpu().numpy() - ref["dE"]) <= 1e-10 * np.linalg.norm(ref["dE"])
    assert abs(got["dw"] - ref["dw"]) <= 1e-10 * max(1.0, abs(ref["dw"]))
    assert abs(got["db"] - ref["db"]) <= 1e-10


# ------------------------------------------------------------------ step kernel: one launch and two launches
STEP_CASES = [
    (300, 7, 64, "clustered"), (257, 5, 128, "clustered"), (700, 9, 256, "random"), (2048, 2, 256, "clustered"),
    (513, 3, 32, "random"), (1024, 10, 256, "clustered"), (256, 20, 256, "clustered"), (260, 40, 128, "random"),
    (4096, 1 + 1, 96, "random"), (129, 10, 256, "clustered"), (200, 5, 64, "random"),
]


@pytest.mark.parametrize("N,M,D,kind", STEP_CASES)
def test_step_kernel_one_launch_vs_oracle(pkg, N, M, D, kind):
    """GE2EPlan.step = prep + ONE step kernel (rows pass, grid barrier, centroid pass) + finalize."""
    assert pkg.lib().ge2e_b200_path(N, N, M, D, 0, 1) == 1
    E_np = orc.make_embeddings(N, M, D, seed=N + 3 * M + D, kind=kind)
    E = torch.tensor(E_np, device=DEV)
    ref = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
    got, plan = run_plan(pkg, E, 10.0, -5.0, "tf32")
    check_dev(got, ref, N * M, TF32_TOL)
    # the two-launch path (module API: forward rows pass, backward centroid pass) gives the same numbers
    two = run_module(pkg, E, 10.0, -5.0, "tf32")
    assert abs(two["loss"] - got["loss"]) <= 1e-6 * abs(got["loss"])
    assert trel(two["dE"], got["dE"]) <= 2e-5          # float atomics: summation order differs between runs
    assert abs(two["dw"] - got["dw"]) <= 1e-4 * max(1.0, abs(got["dw"]))
    # a forward nobody differentiates runs the forward-only kernel: same loss
    with torch.no_grad():
        crit = pkg.GE2ELoss(None, device=E.device, precision="tf32")
        l0 = crit(E).item()
    assert abs(l0 - got["loss"]) <= 1e-5 * abs(got["loss"])


@pytest.mark.parametrize("w,b,g", [(-3.0, 0.5, 0.25), (30.0, -10.0, -1.5), (1.0, 0.0, 1.0), (0.0, 0.3, 1.0)])
def test_step_kernel_scalars(pkg, w, b, g):
    """Negative / large / zero w (s3:22 clamps nothing), upstream gradient != 1 (two-launch path takes g)."""
    N, M, D = 384, 4, 128
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=21, kind="clustered"), device=DEV)
    ref = orct.forward_backward(E, w, b, 1e-6, "softmax", g=g)
    got = run_module(pkg, E, w, b, "tf32", g=g)
    check_dev(got, ref, N * M, TF32_TOL)


def test_step_kernel_repeated_use_of_one_workspace(pkg):
    """The step kernel's counters (zero-fill, pass barrier, exits) are restored by the last CTA: the same
    plan run again and again -- eagerly and as a captured graph over several steps -- repeats its result."""
    N, M, D = 640, 6, 256
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=5, kind="clustered"), device=DEV)
    w = torch.tensor(10.0, device=DEV)
    b = torch.tensor(-5.0, device=DEV)
    plan = pkg.GE2EPlan(N, M, D, "softmax", "tf32", device=DEV)
    outs = []
    for _ in range(3):
        plan.step(E, w, b)
        torch.cuda.synchronize()
        outs.append((plan.loss.item(), plan.dE.clone(), plan.dw.item(), plan.db.item()))
    g = plan.capture(E, w, b, steps=4)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    outs.append((plan.loss.item(), plan.dE.clone(), plan.dw.item(), plan.db.item()))
    for o in outs[1:]:
        assert abs(o[0] - outs[0][0]) <= 1e-6 * abs(outs[0][0])
        assert trel(o[1], outs[0][1]) <= 2e-5
        assert abs(o[2] - outs[0][2]) <= 1e-4 * max(1.0, abs(outs[0][2]))
    assert plan.launches_per_step == 3          # prep, step, finalize


# ------------------------------------------------------------------ full BASELINE sizes against fp64 on the device
@pytest.mark.parametrize("precision,tol", [("fp32", FP32_TOL), ("tf32", TF32_TOL)])
@pytest.mark.parametrize("kind", ["random", "clustered"])
def test_cfg3_full_size_vs_fp64_on_device(pkg, precision, tol, kind):
    N, M, D = 1024, 10, 256
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=33, kind=kind), device=DEV)
    ref = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
    got, _ = run_plan(pkg, E, 10.0, -5.0, precision)
    check_dev(got, ref, N * M, tol)


@pytest.mark.parametrize("precision,tol", [("tf32", TF32_TOL), ("fp32", FP32_TOL)])
def test_cfg4_full_size_vs_fp64_on_device(pkg, precision, tol):
    """BASELINE config 4 (N = 8192, M = 16, D = 256) on one GPU: loss, the whole dE, dw, db against the
    chunked float64 restatement on the same device (1.6 TFLOP of DGEMM: seconds on a B200)."""
    N, M, D = 8192, 16, 256
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=11, kind="clustered"), device=DEV)
    ref = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax", chunk=8192)
    got, _ = run_plan(pkg, E, 10.0, -5.0, precision)
    check_dev(got, ref, N * M, tol)
    if precision == "tf32":
        # per-speaker view: no speaker block of dE is off by more than the tolerance allows for the whole
        err = (got["dE"].double() - ref["dE"]).reshape(N, -1).norm(dim=1)
        nrm = ref["dE"].reshape(N, -1).norm(dim=1)
        assert (err / nrm).max().item() <= 5 * tol


# ------------------------------------------------------------------ speaker shards emulated on one GPU
def run_shards(pkg, E, w, b, R, precision, one_launch, variant=0, g=1.0):
    """Every shard r runs prep / rows / finalize with spk_offset = r * n_local exactly as rank r of a
    speaker-sharded job would; the all-gather is the shared c_hat_all buffer, the reduce-scatter is the sum
    of the full-height partials taken here.  E may be float32, bfloat16 or float16 (dE comes back in E's type);
    g is the upstream gradient.  Returns dict(loss, dE, dw, db) of the whole batch."""
    from speaker_embedding_ge2e_loss_b200 import ops, _lib
    h = pkg.lib()
    N, M, D = E.shape
    nl = N // R
    prec = _lib.PRECISIONS[precision]
    dev = E.device
    wt, bt = torch.tensor(float(w), device=dev), torch.tensor(float(b), device=dev)
    gt = torch.tensor(float(g), device=dev)
    c_hat_all = torch.empty((N, D), device=dev)
    st = []
    for r in range(R):                                   # stage 1 on every shard, then the "all-gather" is complete
        Er = E[r * nl:(r + 1) * nl].contiguous()
        e_hat, cos_diag, accum = ops.prep(Er, c_hat_all[r * nl:(r + 1) * nl], prec)
        st.append(dict(E=Er, e_hat=e_hat, cos_diag=cos_diag, accum=accum))
    dC_sum = torch.zeros((N, D), dtype=torch.float64, device=dev)
    loss = dw = db = 0.0
    for r, s in enumerate(st):
        off = r * nl
        if one_launch:
            U = nl * M
            f32 = dict(dtype=torch.float32, device=dev)
            s["row_stat"], s["row_aux"], s["row_scale"] = torch.empty(U, **f32), torch.empty(U, **f32), torch.empty(U, **f32)
            kst = torch.empty(U, dtype=torch.int32, device=dev)
            s["dE_hat"], dC_part = torch.empty((U, D), **f32), torch.empty((N, D), **f32)
            nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, variant, prec)
            ws = torch.zeros(max(nb, 1), dtype=torch.uint8, device=dev)
            rc = h.ge2e_b200_step_rows(s["e_hat"].data_ptr(), c_hat_all.data_ptr(), s["cos_diag"].data_ptr(), nl, N, off,
                                       M, D, wt.data_ptr(), bt.data_ptr(), 1e-6, variant, prec, gt.data_ptr(),
                                       s["row_stat"].data_ptr(), kst.data_ptr(), s["row_aux"].data_ptr(),
                                       s["row_scale"].data_ptr(), s["accum"].data_ptr(), s["dE_hat"].data_ptr(),
                                       dC_part.data_ptr(), ws.data_ptr() if nb else None, nb,
                                       torch.cuda.current_stream().cuda_stream)
            assert rc == 0, h.ge2e_b200_strerror(rc)
            if not (h.ge2e_b200_path(nl, N, M, D, variant, prec) in (1, 2, 3) and variant == 0):
                s["row_scale"] = None
            torch.cuda.synchronize()
            assert not ws[:256].any(), "the workspace's counters must be zero again after the call"
            dwdb = s["accum"][1:3]
        else:
            rs, ks, aux, _, _, dE_hat, row_scale = ops.fwd_rows(s["e_hat"], c_hat_all, s["cos_diag"], nl, N, off, M, D,
                                                                wt, bt, 1e-6, variant, prec, s["accum"], want_grad=True)
            s["dE_hat"], dC_part, dwdb = ops.bwd_rows(s["e_hat"], c_hat_all, s["cos_diag"], rs, ks, aux, nl, N, off, M,
                                                      D, wt, bt, 1e-6, variant, prec, gt, dE_hat=dE_hat,
                                                      row_scale=row_scale)
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
                                   1e-6, variant, gt, row_scale=s["row_scale"]))
    torch.cuda.synchronize()
    return dict(loss=loss, dE=torch.cat(dE, dim=0), dw=dw, db=db)


@pytest.mark.parametrize("N,M,D,R,precision,tol", [
    (64, 10, 256, 2, "fp32", FP32_TOL), (512, 4, 256, 4, "fp32", FP32_TOL), (96, 5, 64, 3, "fp32", FP32_TOL),
    (512, 4, 256, 2, "tf32", TF32_TOL), (1024, 10, 256, 8, "tf32", TF32_TOL), (768, 3, 128, 3, "tf32", TF32_TOL),
    (2048, 8, 256, 8, "tf32", TF32_TOL),
    # fp32-class on the tensor cores: a centroid row carries its hi and lo fp16 planes through the "all-gather"
    (1024, 10, 256, 8, "fp32_split", FP32_TOL), (768, 3, 128, 3, "fp32_split", FP32_TOL),
    (2048, 8, 256, 2, "fp32_split", FP32_TOL),
])
@pytest.mark.parametrize("one_launch", [False, True])
def test_speaker_shards_on_one_gpu_vs_oracle(pkg, N, M, D, R, precision, tol, one_launch):
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + R, kind="clustered"), device=DEV)
    if precision == "tf32":
        assert pkg.lib().ge2e_b200_path(N // R, N, M, D, 0, 1) == 1, "the shard should take the tcgen05 path"
    if precision == "fp32_split":
        assert pkg.lib().ge2e_b200_path(N // R, N, M, D, 0, 2) == 2, "the shard should take the split tcgen05 path"
    ref = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
    got = run_shards(pkg, E, 10.0, -5.0, R, precision, one_launch)
    check_dev(got, ref, N * M, tol)


# ------------------------------------------------------------------ contrast loss on the tensor-core forward
def test_cfg3_contrast_tf32_gradients_on_robust_rows(pkg):
    """The contrast gradient has two non-zeros per row (own centroid, hardest negative).  TF32 rounding of
    the similarities can swap two near-tied negatives; on every row whose top-2 gap exceeds the TF32
    perturbation of S the arg-max -- hence the row of dE_hat -- must agree with float64."""
    N, M, D = 1024, 10, 256
    w, b = 10.0, -5.0
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=4, kind="random"), device=DEV)
    ref = orct.forward_backward(E, w, b, 1e-6, "contrast")
    got = run_module(pkg, E, w, b, "tf32", variant="contrast")
    assert abs(got["loss"] - ref["loss"]) <= TF32_TOL * abs(ref["loss"])
    ok = robust_speakers(E, w)
    err = trel(got["dE"][ok], ref["dE"][ok].float())
    assert err <= TF32_TOL, err
    assert abs(got["dw"] - ref["dw"]) <= 2e-2 * max(1.0, abs(ref["dw"]))


def robust_speakers(E, w):
    """Mask of the speakers whose contrast gradient TF32 rounding cannot change: all their rows have a robust
    arg-max and they are no fragile row's own or hardest-negative speaker."""
    N, M, D = E.shape
    dev = E.device
    # rows with a robust arg-max: top-2 gap of the negatives' cosines > 2e-4 (TF32 cos error ~ 1e-5 rms at D = 256)
    E64 = E.double()
    Eh = torch.nn.functional.normalize(E64.reshape(N * M, D), dim=1)
    Ch = torch.nn.functional.normalize(E64.mean(1), dim=1)
    S = w * (Eh @ Ch.T)
    rows = torch.arange(N * M, device=dev)
    S[rows, rows // M] = -float("inf")
    top2 = S.topk(2, dim=1).values
    robust = (top2[:, 0] - top2[:, 1]) > 2e-4 * abs(w)
    assert robust.float().mean().item() > 0.95
    # speakers all of whose rows are robust AND that are nobody's fragile arg-max get the exact gradient
    fragile_rows = ~robust
    touched = torch.zeros(N, dtype=torch.bool, device=dev)
    touched[(rows // M)[fragile_rows]] = True
    top1 = S.topk(2, dim=1).indices
    touched[top1[fragile_rows].reshape(-1)] = True
    ok = ~touched
    assert ok.float().mean().item() > 0.5
    return ok


# ------------------------------------------------------------------ TF32 step with MMA1 on fp16 copies of the operands
@pytest.mark.parametrize("N,M,D", [(300, 7, 128), (1024, 10, 256), (700, 9, 192), (513, 3, 64)])
def test_hybrid_operand_copies_match_the_tf32_step(pkg, N, M, D):
    """Large shapes (>= 2^26 utterance x speaker pairs: config 4, covered by the full-size test above) run the first
    product of the TF32 step on fp16 copies of e_hat / c_hat made by a conversion launch (ge2e_b200_debug_hybrid).
    Forced on small shapes here: same tolerance class, results next to the plain TF32 step's, one more launch,
    workspace counters restored; a speaker shard takes the same path."""
    h = pkg.lib()
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + D, kind="clustered"), device=DEV)
    ref = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
    plain, _ = run_plan(pkg, E, 10.0, -5.0, "tf32")
    h.ge2e_b200_debug_hybrid(1)
    try:
        got, plan = run_plan(pkg, E, 10.0, -5.0, "tf32")
        w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
        g = plan.capture(E, w, b, steps=2)
        g.replay()
        torch.cuda.synchronize()
        assert plan.launches_per_step == 4          # prep, conversion, step, finalize
        assert int(plan._ws[:256].max()) == 0
        again = dict(loss=plan.loss.item(), dE=plan.dE.clone(), dw=plan.dw.item(), db=plan.db.item())
        shards = run_shards(pkg, E, 10.0, -5.0, 3 if N % 3 == 0 else 1, "tf32", True)
    finally:
        h.ge2e_b200_debug_hybrid(0)
    for r in (got, again, shards):
        check_dev(r, ref, N * M, TF32_TOL)
    assert trel(got["dE"], ref["dE"]) <= 2 * trel(plain["dE"], ref["dE"]) + 1e-6
