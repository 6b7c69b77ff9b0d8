"""bfloat16 / float16 embeddings through every public path.

The contract (include/ge2e_b200.h, ge2e_dtype): E is widened to fp32 when it is loaded, so every number after that
load is the one the fp32 call computes for E.float(); dE has E's dtype and is rounded to it once, after the upstream
gradient has been applied.  So each kernel family is checked against (a) the fp32 call on E.float() on the same
path -- loss and dw to 1e-6, every dE element within one ulp of E's dtype -- and (b) the float64 oracle on
E.double(), with the rounding of dE (2^-8 bf16, 2^-11 fp16) added to the path's tolerance.  Every case asserts which
path ran (plan.path, plan.single_kernel), as test_gpu_edges.py does.
"""
import os
import subprocess
import sys
import textwrap

import pytest
import torch

from oracle import ge2e_oracle as orc
from test_gpu_edges import (DEV, FP32_TOL, TF32_TOL, check, pkg, reference, run_module, run_unperm,  # noqa: F401
                            small_step_mode, trel)

pytestmark = pytest.mark.gpu

HALF = [torch.bfloat16, torch.float16]
ROUND = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}       # relative rounding of one dE element
MANT = {torch.bfloat16: 7, torch.float16: 10}                        # stored mantissa bits
EMIN = {torch.bfloat16: -126, torch.float16: -14}                    # smallest normal exponent
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ulp(x, dtype):
    """Spacing of dtype's values at |x| (subnormal spacing below the normal range)."""
    e = torch.floor(torch.log2(x.double().abs().clamp_min(1e-300))).clamp_min(EMIN[dtype])
    return torch.exp2(e - MANT[dtype])


# The centroid-gradient sums (and, on the tensor-core paths, the softmax row sums) are accumulated in no fixed order,
# so two fp32 runs of the same step already differ: in the last bits on the SIMT paths, at the operand rounding of
# TF32 / fp16 on the tensor-core paths.  An element that is the small difference of large terms can move by that
# much in absolute terms, more than one ulp of its own small magnitude; SLACK (relative to the largest |dE|) is
# that run-to-run spread, allowed on top of the ulp.
SLACK = {0: 1e-5, 1: 2e-3, 2: 1e-5, 3: 2e-3}


def assert_within_one_ulp(got, ref32, dtype, path=0):
    """|got - ref32| <= one ulp of dtype (the spacing at the larger of the two: a value next to a power of two may
    round across it) + the reference's own run-to-run spread."""
    assert got.dtype == dtype
    d = (got.double() - ref32.double()).abs()
    slack = SLACK[path] * ref32.double().abs().max()
    bad = d > ulp(torch.maximum(got.double().abs(), ref32.double().abs()), dtype) + slack
    assert not bad.any(), (int(bad.sum()), d.max().item())


def half_batch(N, M, D, dtype, kind="clustered"):
    return torch.tensor(orc.make_embeddings(N, M, D, seed=N + M + D, kind=kind), device=DEV).to(dtype)


def run_plan_dtype(pkg, E, precision, variant, w=10.0, b=-5.0):
    N, M, D = E.shape
    plan = pkg.GE2EPlan(N, M, D, variant, precision, device=E.device, dtype=E.dtype)
    wt, bt = torch.tensor(float(w), device=E.device), torch.tensor(float(b), device=E.device)
    plan.step(E, wt, bt)
    torch.cuda.synchronize()
    return dict(loss=plan.loss.item(), dE=plan.dE.clone(), dw=plan.dw.item(), db=plan.db.item()), plan


def check_against_fp32(got, ref32, U, dtype, path):
    assert abs(got["loss"] - ref32["loss"]) <= 1e-6 * max(1.0, abs(ref32["loss"])), (got["loss"], ref32["loss"])
    assert abs(got["dw"] - ref32["dw"]) <= 1e-6 * max(1.0, abs(ref32["dw"])), (got["dw"], ref32["dw"])
    assert abs(got["db"] - ref32["db"]) <= 1e-6 * U, (got["db"], ref32["db"])
    assert_within_one_ulp(got["dE"], ref32["dE"].reshape(got["dE"].shape), dtype, path)
    assert trel(got["dE"].float(), ref32["dE"]) <= ROUND[dtype] + SLACK[path]


# (N, M, D, precision, variant, small-step mode, expected path, expected single kernel)
CASES = [
    (4, 8, 256, "fp32", "softmax", 1, 0, True),          # the single-kernel step, reference test shape
    (64, 10, 256, "fp32", "softmax", 1, 0, True),        # ... reference training shape
    (64, 10, 256, "fp32", "softmax", 0, 0, False),       # the SIMT pipeline (register prep / finalize)
    (129, 10, 256, "tf32", "softmax", 1, 1, False),      # tcgen05 TF32
    (129, 10, 256, "fp32", "softmax", 1, 2, False),      # the default fp32: split fp16 planes
    (129, 10, 256, "f16", "softmax", 1, 3, False),       # one fp16 plane
    (129, 10, 128, "fp32", "softmax", 1, 2, False),      # the default at D = 128
    (7, 10, 256, "fp32", "contrast", 0, 0, False),       # contrast, last block with one speaker
    (129, 10, 256, "fp32", "contrast", 0, 0, False),
    (8, 10, 512, "fp32", "softmax", 0, 0, False),        # D = 512: the warp kernels
    (8, 20, 256, "fp32", "softmax", 0, 0, False),        # M = 20: warp, not register kernels
    (6, 40, 256, "fp32", "softmax", 0, 0, False),        # M = 40: the generic (shared-memory) finalize
    (8, 10, 100, "fp32", "softmax", 1, 0, True),         # D = 100: generic bodies inside the single kernel
    (8, 10, 100, "fp32", "softmax", 0, 0, False),        # ... and the generic prep / finalize kernels
]


@pytest.mark.parametrize("dtype", HALF, ids=["bf16", "fp16"])
@pytest.mark.parametrize("N,M,D,precision,variant,mode,path,single", CASES)
def test_every_kernel_family(pkg, dtype, N, M, D, precision, variant, mode, path, single):
    E = half_batch(N, M, D, dtype)
    with small_step_mode(pkg, mode):
        got, plan = run_plan_dtype(pkg, E, precision, variant)
        ref32, plan32 = run_plan_dtype(pkg, E.float(), precision, variant)
    assert plan.path == plan32.path == path and plan.single_kernel == plan32.single_kernel == single
    assert got["dE"].dtype == dtype and ref32["dE"].dtype == torch.float32
    check_against_fp32(got, ref32, N * M, dtype, path)
    tol = (TF32_TOL if path in (1, 3) else FP32_TOL) + ROUND[dtype]
    check(dict(got, dE=got["dE"].float()), reference(E.double().cpu().numpy(), 10.0, -5.0, variant), N * M, tol)


@pytest.mark.parametrize("N,precision", [(64, "fp32"), (129, "fp32"), (129, "tf32")])
def test_unperm_matches_plain_call(pkg, N, precision):
    E = half_batch(N, 10, 256, torch.bfloat16)
    plain = run_module(pkg, E, 10.0, -5.0, precision, "softmax")
    shuffled = run_unperm(pkg, E, 10.0, -5.0, precision, "softmax", seed=N)
    assert shuffled["dE"].dtype == torch.bfloat16
    assert abs(plain["loss"] - shuffled["loss"]) <= 1e-6 * abs(plain["loss"])
    assert abs(plain["dw"] - shuffled["dw"]) <= 1e-6 * max(1.0, abs(plain["dw"]))
    assert_within_one_ulp(shuffled["dE"], plain["dE"].float(), torch.bfloat16, 1 if precision == "tf32" else 0)


def at_offset(E, off):
    """E's values in fresh storage, `off` elements past the start of the allocation (not 8-byte aligned)."""
    buf = torch.zeros(E.numel() + 8, dtype=E.dtype, device=E.device)
    out = buf[off:off + E.numel()].view(E.shape)
    out.copy_(E)
    return out


@pytest.mark.parametrize("dtype", HALF, ids=["bf16", "fp16"])
@pytest.mark.parametrize("precision,path", [("fp32", 2), ("fp32_simt", 0)])
def test_unaligned_inputs(pkg, dtype, precision, path):
    E = half_batch(129, 10, 256, dtype)
    crit = pkg.GE2ELoss(None, device=E.device, precision=precision)
    assert crit.path_for(129, 10, 256) == path
    aligned = run_module(pkg, E, 10.0, -5.0, precision, "softmax")
    for off in (1, 2, 3):
        Eo = at_offset(E, off)
        assert Eo.data_ptr() % 8 != 0
        got = run_module(pkg, Eo, 10.0, -5.0, precision, "softmax")
        assert abs(got["loss"] - aligned["loss"]) <= 1e-6 * abs(aligned["loss"])
        assert_within_one_ulp(got["dE"], aligned["dE"].float(), dtype, path)
        if path == 2:
            plan = pkg.GE2EPlan(129, 10, 256, precision=precision, device=E.device, dtype=dtype)
            with pytest.raises(ValueError, match="aligned"):
                plan.step(Eo, torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV))


@pytest.mark.parametrize("N,precision", [(64, "fp32"), (129, "tf32")])
def test_bf16_plan_eager_and_graph(pkg, N, precision):
    M, D, dt = 10, 256, torch.bfloat16
    Es = [half_batch(N, M, D, dt), (half_batch(N, M, D, dt).float() * 1.5 + 0.25).to(dt)]
    w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
    plan = pkg.GE2EPlan(N, M, D, "softmax", precision, device=DEV, dtype=dt)
    plan32 = pkg.GE2EPlan(N, M, D, "softmax", precision, device=DEV)
    g = plan.capture(Es, w, b, steps=2)             # step 0 on Es[0], step 1 on Es[1]
    plan32.capture([e.float() for e in Es], w, b, steps=2)
    assert plan.launches_per_step == plan32.launches_per_step
    for replay in (True, False):
        if replay:
            g.replay()
        else:
            plan.step(Es[1], w, b)
        torch.cuda.synchronize()
        ref = run_module(pkg, Es[1], 10.0, -5.0, precision, "softmax")
        assert plan.dE.dtype == dt
        assert abs(plan.loss.item() - ref["loss"]) <= 1e-6 * abs(ref["loss"])
        assert abs(plan.dw.item() - ref["dw"]) <= 1e-6 * max(1.0, abs(ref["dw"]))
        assert_within_one_ulp(plan.dE, ref["dE"].float(), dt, plan.path)
    with pytest.raises(TypeError, match="bfloat16"):
        plan.step(Es[0].float(), w, b)


# ------------------------------------------------------------------ fp16 and loss scaling
def scaled_speaker_batch(N=64, M=10, D=256, speaker=3, factor=3e4):
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=5, kind="clustered"), device=DEV)
    E = E / E.norm(dim=-1, keepdim=True)
    Es = E.clone()
    Es[speaker] *= factor
    return E.half(), Es.half(), speaker


def test_fp16_gradients_survive_loss_scaling(pkg):
    from speaker_embedding_ge2e_loss_b200 import _lib, ops
    E, Es, j = scaled_speaker_batch()
    scale = 2.0 ** 16
    base = run_module(pkg, E, 10.0, -5.0, "fp32", "softmax")
    ref = reference(Es.double().cpu().numpy(), 10.0, -5.0, "softmax")
    ref_j = ref["dE"][j] * scale
    # cosines are scale invariant: same loss; that speaker's gradient shrinks by the factor, into fp16 subnormals
    one = run_module(pkg, Es, 10.0, -5.0, "fp32", "softmax")
    assert abs(one["loss"] - base["loss"]) <= 1e-5 * abs(base["loss"])
    assert ref["dE"][j].abs().max().item() < 2.0 ** -14
    # rounding to fp16 first and scaling afterwards loses the speaker's gradient: the test can tell the difference
    assert trel(one["dE"][j].double() * scale, ref_j) > 2.0 ** -10
    # eager path (step in forward, scaling in backward) and custom-op path (upstream gradient inside finalize)
    eager = run_module(pkg, Es, 10.0, -5.0, "fp32", "softmax", g=scale)
    Eg = Es.clone().requires_grad_(True)
    w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
    vcode = _lib.VARIANTS["softmax"]
    pcode = _lib.resolve_precision("fp32", 64, 64, 10, 256, vcode)
    loss = ops.ge2e_fwd(Eg, w, b, 1e-6, vcode, pcode)[0]
    loss.backward(torch.tensor(scale, device=DEV))
    for dE in (eager["dE"], Eg.grad):
        assert dE.dtype == torch.float16 and torch.isfinite(dE[j]).all()
        assert trel(dE[j].double(), ref_j) <= 2.0 ** -10


def test_gradscaler_round_trip(pkg):
    E, Es, j = scaled_speaker_batch()
    crit = pkg.GE2ELoss(None, device=DEV)
    ref = reference(Es.double().cpu().numpy(), 10.0, -5.0, "softmax")
    # 2^12 keeps every speaker's scaled gradient inside fp16's range; 2^30 does not
    for init_scale, finite in ((2.0 ** 12, True), (2.0 ** 30, False)):
        scaler = torch.amp.GradScaler("cuda", init_scale=init_scale)
        leaf = Es.clone().requires_grad_(True)
        scaler.scale(crit(leaf)).backward()
        crit.zero_grad()
        grad = leaf.grad
        assert grad.dtype == torch.float16 and not torch.isnan(grad).any()
        found_inf = torch.zeros(1, device=DEV)
        torch._amp_foreach_non_finite_check_and_unscale_([grad.clone()], found_inf,
                                                         torch.full((1,), 1.0 / init_scale, device=DEV))
        if finite:
            assert torch.isfinite(grad).all() and found_inf.item() == 0.0
            assert trel(grad.double() / init_scale, ref["dE"]) <= FP32_TOL + ROUND[torch.float16]
            assert trel(grad[j].double() / init_scale, ref["dE"][j]) <= 2.0 ** -10
        else:
            assert torch.isinf(grad).any() and found_inf.item() == 1.0


# ------------------------------------------------------------------ host side: no hidden casts, same launches
def test_no_hidden_casts(pkg):
    from torch.profiler import ProfilerActivity, profile
    crit = pkg.GE2ELoss(None, device=DEV)
    base = half_batch(64, 10, 256, torch.bfloat16)
    counts = {}
    for dt in (torch.float32, torch.bfloat16):
        E = base.to(dt).requires_grad_(True)
        crit(E).backward()                               # warm-up: plans, workspaces
        torch.cuda.synchronize()
        E.grad = None
        n0 = pkg.lib().ge2e_b200_launch_count()
        with profile(activities=[ProfilerActivity.CPU]) as prof:
            crit(E).backward()
            torch.cuda.synchronize()
        launches = pkg.lib().ge2e_b200_launch_count() - n0
        names = [ev.name for ev in prof.events()]
        counts[dt] = (names.count("aten::_to_copy"), names.count("aten::copy_"), launches)
        assert E.grad.dtype == dt
    assert counts[torch.bfloat16][0] == 0, counts
    assert counts[torch.bfloat16][1] <= counts[torch.float32][1], counts
    assert counts[torch.bfloat16][2] == counts[torch.float32][2], counts


@pytest.mark.parametrize("unperm", [False, True])
def test_torch_compile(pkg, unperm):
    from speaker_embedding_ge2e_loss_b200 import ge2e_loss
    N, M, D = 64, 10, 256
    E = half_batch(N, M, D, torch.bfloat16)
    w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
    if unperm:
        perm = torch.randperm(N * M, generator=torch.Generator().manual_seed(1)).to(DEV)
        idx = torch.empty_like(perm)
        idx[perm] = torch.arange(N * M, device=DEV)
        E = E.reshape(N * M, D)[perm].contiguous()

        def fn(x, w, b):
            return ge2e_loss(x, w, b, unperm=idx, speakers=N)
    else:
        def fn(x, w, b):
            return ge2e_loss(x, w, b)
    compiled = torch.compile(fn, backend="aot_eager", fullgraph=True)
    out = {}
    for name, f in (("eager", fn), ("compiled", compiled)):
        x = E.clone().requires_grad_(True)
        ww, bb = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        loss = f(x, ww, bb)
        loss.backward()
        torch.cuda.synchronize()
        out[name] = (loss.item(), x.grad.clone(), ww.grad.item())
    assert out["compiled"][1].dtype == torch.bfloat16
    assert abs(out["compiled"][0] - out["eager"][0]) <= 1e-6 * abs(out["eager"][0])
    assert abs(out["compiled"][2] - out["eager"][2]) <= 1e-6 * max(1.0, abs(out["eager"][2]))
    assert_within_one_ulp(out["compiled"][1], out["eager"][1].float(), torch.bfloat16)


SHARDED_CHILD = textwrap.dedent("""
    import os, sys
    import torch, torch.distributed as dist
    sys.path.insert(0, %r)
    import speaker_embedding_ge2e_loss_b200 as pkg
    from oracle import ge2e_oracle as orc
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29579", RANK="0", WORLD_SIZE="1")
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda:0"))
    dev = torch.device("cuda:0")
    for (N, precision) in [(64, "fp32"), (129, "tf32")]:
        E = torch.tensor(orc.make_embeddings(N, 10, 256, seed=N, kind="clustered"), device=dev).bfloat16()
        res = []
        for group in (dist.group.WORLD, None):
            crit = pkg.GE2ELoss(None, device=dev, precision=precision, process_group=group)
            x = E.clone().requires_grad_(True)
            loss = crit(x)
            loss.backward()
            torch.cuda.synchronize()
            res.append((loss.item(), x.grad.double(), crit.w.grad.item()))
        (l0, g0, w0), (l1, g1, w1) = res
        tol = 1e-5 if precision == "fp32" else 2e-3
        rel = ((g0 - g1).norm() / g1.norm()).item()
        assert x.grad.dtype == torch.bfloat16
        assert abs(l0 - l1) <= tol * abs(l1) and abs(w0 - w1) <= tol * max(1.0, abs(w1)), (N, l0, l1, w0, w1)
        assert rel <= tol + 2.0 ** -8, (N, rel)
    print("SHARDED_BF16_OK", flush=True)
    os._exit(0)
""") % ROOT


def test_sharded_autograd_bf16():
    """GE2ELoss(process_group=...) on a world-1 NCCL group (the staged prep / finalize with bf16 E) against the
    single-device module; in a child process with a timeout, as test_gpu_sharded_plan.py."""
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-c", SHARDED_CHILD], capture_output=True, text=True, timeout=300, env=env)
    assert "SHARDED_BF16_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_parameters_must_be_float32(pkg):
    E = half_batch(4, 8, 256, torch.bfloat16)
    for w, b, name in ((torch.tensor(10.0, device=DEV, dtype=torch.bfloat16), torch.tensor(-5.0, device=DEV), "w"),
                       (torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV, dtype=torch.bfloat16), "b")):
        with pytest.raises(TypeError, match=f"^{name} must be float32"):
            pkg.ge2e_loss(E, w, b)


def test_out_of_scope_paths_refuse_half_embeddings(pkg):
    feed = pkg.GE2EHostFeed(4, 8, 256, torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV), depth=1)
    with pytest.raises(ValueError, match="float32 embeddings only"):
        feed.submit(torch.zeros(4, 8, 256, dtype=torch.bfloat16).pin_memory())
