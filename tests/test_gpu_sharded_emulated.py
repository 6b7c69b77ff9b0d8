"""The speaker-sharded step at 2..8 ranks emulated on ONE GPU, against the float64 oracle.

  * Peer memory: ``ShardedGE2EPlan._step_peer`` for every rank r = 0 .. R-1.  The entry points take host arrays of
    plain device pointers, so every rank's buffers live on this GPU; the ranks run one after another on one stream
    (never on concurrent streams: the step kernel's pass 2 needs its whole grid co-resident, two overlapping step
    kernels could wait on each other), and a device synchronise stands where the plan has its two cross-rank
    barriers.  Up to config 4 on 8 ranks, where the step takes the fp16-operand-copy (HYB) kernel and pass 2
    reduce-adds into the owners' rows.
  * The inputs ``ge2e_b200_step_rows_peers`` and ``ge2e_b200_peer_publish`` refuse: the error code, no launch, no
    byte of any buffer changed.
  * The reduce-scatter path (``run_shards``) with the contrast loss, bfloat16 / float16 embeddings and an upstream
    gradient other than 1.
"""
import ctypes as C

import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_oracle_torch as orct
from test_gpu_step import DEV, FP32_TOL, TF32_TOL, check_dev, pkg, robust_speakers, run_shards, trel  # noqa: F401

pytestmark = pytest.mark.gpu

EPS = 1e-6
W, B = 10.0, -5.0
OK, SHAPE, UNSUPPORTED, ARGUMENT = 0, -1, -2, -3
SOFTMAX, CONTRAST = 0, 1
FP32, TF32, FP32_SPLIT, F16 = 0, 1, 2, 3
NAME = {TF32: "tf32", FP32_SPLIT: "fp32_split", F16: "f16"}      # the precision code's name for run_shards
PATH = {TF32: 1, FP32_SPLIT: 2, F16: 3}


def ptrs(ps):
    return (C.c_void_p * len(ps))(*ps)


def check_rc(h, rc, what):
    assert rc == OK, f"{what}: {h.ge2e_b200_strerror(rc).decode()}"


def hybrid_selected(h, nl, N, M, D, mode=0):
    """Whether the TF32 step takes the fp16 operand copies (HYB) under ge2e_b200_debug_hybrid(mode): the copies
    live in the workspace, which is then larger than with them switched off.  Leaves the default mode (0) set."""
    try:
        h.ge2e_b200_debug_hybrid(mode)
        now = h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, TF32)
        h.ge2e_b200_debug_hybrid(-1)
        plain = h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, TF32)
    finally:
        h.ge2e_b200_debug_hybrid(0)
    return now > plain


# ------------------------------------------------------------------ peer-memory step, R ranks on one GPU
def run_peers(pkg, E, w, b, R, prec, g=1.0):
    """prep -> publish c_hat slice + clear dC_local -> [barrier] -> step_rows_peers -> publish {loss, dw, db} ->
    [barrier] -> finalize -> sum of the table, for every rank.  Checks the exchange itself (c_hat_all replicas
    bit-identical, NaN canaries between the ranks' buffers untouched, workspace counters zero again) and returns
    dict(loss, dE, dw, db) of the whole batch and the launches of one step_rows_peers call."""
    h = pkg.lib()
    N, M, D = E.shape
    nl = N // R
    U = nl * M
    dev = E.device
    f32 = dict(dtype=torch.float32, device=dev)
    wt, bt, gt = (torch.tensor(float(v), **f32) for v in (w, b, g))
    s = torch.cuda.current_stream().cuda_stream
    nan = float("nan")
    # every rank's c_hat_all [N, D] in one tensor and every rank's dC_local [nl, D] in another, with a NaN row in
    # front of, between and behind them (D % 32 == 0: every slice starts 16-byte aligned)
    c_buf = torch.full((R * (N + 1) + 1, D), nan, **f32)
    d_buf = torch.full((R * (nl + 1) + 1, D), nan, **f32)
    c_all = [c_buf[1 + r * (N + 1):1 + r * (N + 1) + N] for r in range(R)]
    dC = [d_buf[1 + r * (nl + 1):1 + r * (nl + 1) + nl] for r in range(R)]
    c_canary = torch.arange(R + 1, device=dev) * (N + 1)
    d_canary = torch.arange(R + 1, device=dev) * (nl + 1)
    tables = torch.full((R, R, 4), nan, **f32)                 # [rank q's copy][row of rank r]
    nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, prec)
    assert nb > 0
    ranks = []
    for r in range(R):
        ranks.append(dict(E=E[r * nl:(r + 1) * nl], e_hat=torch.empty((U, D), **f32), cos_diag=torch.empty(U, **f32),
                          accum=torch.empty(4, **f32), row_stat=torch.empty(U, **f32), row_aux=torch.empty(U, **f32),
                          row_kstar=torch.empty(U, dtype=torch.int32, device=dev), row_scale=torch.empty(U, **f32),
                          dE_hat=torch.empty((U, D), **f32), dE=torch.empty((nl, M, D), **f32),
                          ws=torch.zeros(nb, dtype=torch.uint8, device=dev)))
    for r, k in enumerate(ranks):                           # 1. prep into the rank's own slice
        check_rc(h, h.ge2e_b200_prep(k["E"].data_ptr(), nl, M, D, prec, k["e_hat"].data_ptr(),
                                     c_all[r][r * nl:].data_ptr(), k["cos_diag"].data_ptr(), k["accum"].data_ptr(), s),
                 "ge2e_b200_prep")
    for r in range(R):                                      # 2. the slice into every peer's c_hat_all; clear dC_local
        off = r * nl * D * 4
        peers = ptrs([c_all[q].data_ptr() + off for q in range(R) if q != r])
        check_rc(h, h.ge2e_b200_peer_publish(c_all[r][r * nl:].data_ptr(), peers, R - 1, 0, nl * D, dC[r].data_ptr(),
                                             nl * D, s), "ge2e_b200_peer_publish")
    torch.cuda.synchronize()                                # barrier 1
    owners = ptrs([d.data_ptr() for d in dC])
    launches = set()
    for r, k in enumerate(ranks):                           # 3. the step; pass 2 adds into the owners' rows
        n0 = h.ge2e_b200_launch_count()
        check_rc(h, h.ge2e_b200_step_rows_peers(k["e_hat"].data_ptr(), c_all[r].data_ptr(), k["cos_diag"].data_ptr(),
                                                nl, N, r * nl, M, D, wt.data_ptr(), bt.data_ptr(), EPS, SOFTMAX, prec,
                                                gt.data_ptr(), k["row_stat"].data_ptr(), k["row_kstar"].data_ptr(),
                                                k["row_aux"].data_ptr(), k["row_scale"].data_ptr(),
                                                k["accum"].data_ptr(), k["dE_hat"].data_ptr(), owners, R,
                                                k["ws"].data_ptr(), nb, s), "ge2e_b200_step_rows_peers")
        launches.add(h.ge2e_b200_launch_count() - n0)
        torch.cuda.synchronize()
        assert not k["ws"][:256].any(), f"rank {r}: the workspace's counters must be zero again after the call"
    for r, k in enumerate(ranks):                           # 4. {loss, dw, db} into row r of every rank's table
        rows = ptrs([tables[q, r].data_ptr() for q in range(R)])
        check_rc(h, h.ge2e_b200_peer_publish(k["accum"].data_ptr(), rows, R, 0, 4, None, 0, s),
                 "ge2e_b200_peer_publish")
    torch.cuda.synchronize()                                # barrier 2
    for r, k in enumerate(ranks):                           # 5. finalize on the rank's own dC_local
        check_rc(h, h.ge2e_b200_bwd_finalize(k["E"].data_ptr(), k["dE_hat"].data_ptr(), dC[r].data_ptr(),
                                             k["cos_diag"].data_ptr(), k["row_stat"].data_ptr(),
                                             k["row_aux"].data_ptr(), k["row_scale"].data_ptr(), nl, M, D,
                                             wt.data_ptr(), bt.data_ptr(), EPS, SOFTMAX, gt.data_ptr(),
                                             k["dE"].data_ptr(), s), "ge2e_b200_bwd_finalize")
    sums = tables.sum(dim=1)                                # 6. every rank sums its own table
    torch.cuda.synchronize()

    # GE2E_F16 rows hold the hi fp16 plane alone: prep writes the first half of each row's bytes
    written = D // 2 if prec == F16 else D
    assert not c_all[0][:, :written].isnan().any(), "a slice of c_hat_all was never published"
    for r in range(1, R):
        assert unchanged([c_all[0]], [c_all[r]]), f"rank {r}'s c_hat_all differs from rank 0's"
        assert torch.equal(tables[r], tables[0]), f"rank {r}'s scalar table differs from rank 0's"
    assert c_buf[c_canary].isnan().all() and d_buf[d_canary].isnan().all(), "a write left its rank's buffer"
    assert len(launches) == 1, launches
    loss, dw, db = sums[0, :3].tolist()
    return dict(loss=loss, dE=torch.cat([k["dE"] for k in ranks]), dw=dw, db=db, launches=launches.pop())


@pytest.fixture(scope="module")
def cfg4():
    """BASELINE config 4 and its float64 reference (w = 10, b = -5, g = 1): computed once for every cfg4 case."""
    E = torch.tensor(orc.make_embeddings(8192, 16, 256, seed=11, kind="clustered"), device=DEV)
    return E, orct.forward_backward(E, W, B, EPS, "softmax", chunk=8192)


# (N, M, D, ranks, precision, HYB selected, w, upstream gradient)
PEER_CASES = [
    (256, 6, 128, 2, "tf32", False, W, 1.0),            # peer_rows = 128: one owner tile per rank
    (256, 6, 96, 2, "tf32", False, W, 1.0),             # D / 32 odd: CTA size 1 (pick_cg)
    (1024, 6, 256, 2, "tf32", False, W, 1.0),           # the 2-GPU test's shape
    (1024, 6, 256, 2, "fp32", False, W, 1.0),
    (1024, 6, 256, 2, "tf32", False, -3.0, -1.5),       # negative w, upstream gradient through grad_out
    (768, 4, 256, 3, "tf32", False, W, 1.0),            # odd rank count
    (2048, 8, 256, 4, "tf32", False, W, 1.0),
    (2048, 8, 256, 4, "fp32", False, W, 1.0),
    (2048, 8, 256, 4, "fp32", False, -3.0, -1.5),
    (1024, 10, 256, 8, "tf32", False, W, 1.0),          # 8 ranks, one owner tile per rank
    (1024, 10, 256, 8, "fp32", False, W, 1.0),
    (1024, 10, 256, 8, "f16", False, W, 1.0),
    (8192, 16, 256, 8, "tf32", True, W, 1.0),           # config 4 on 8 ranks: HYB + peers, the headline instantiation
    (8192, 16, 256, 8, "fp32", False, W, 1.0),
    (8192, 16, 256, 2, "tf32", True, W, 1.0),           # HYB + peers, 2 ranks
]


@pytest.mark.parametrize("N,M,D,R,precision,hyb,w,g", PEER_CASES)
def test_peer_memory_step_emulated_vs_oracle(pkg, request, N, M, D, R, precision, hyb, w, g):
    from speaker_embedding_ge2e_loss_b200 import _lib
    h = pkg.lib()
    nl = N // R
    prec = _lib.resolve_precision(precision, nl, N, M, D, SOFTMAX)
    assert prec == {"tf32": TF32, "fp32": FP32_SPLIT, "f16": F16}[precision]
    assert h.ge2e_b200_path(nl, N, M, D, SOFTMAX, prec) == PATH[prec]
    if prec == TF32:
        assert hybrid_selected(h, nl, N, M, D) == hyb
    if (N, M, D) == (8192, 16, 256):
        assert w == W and g == 1.0
        E, ref = request.getfixturevalue("cfg4")
    else:
        E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + M + R, kind="clustered"), device=DEV)
        ref = orct.forward_backward(E, w, B, EPS, "softmax", g=g)
    got = run_peers(pkg, E, w, B, R, prec, g)
    # one step kernel; the plane precisions' forward kernel, the HYB conversion ahead of it
    assert got["launches"] == 1 + (prec != TF32) + hyb
    tol = FP32_TOL if prec == FP32_SPLIT else TF32_TOL
    check_dev(got, ref, N * M, tol)
    # the reduce-scatter path on the same batch: the same numbers up to the order of the float atomics
    rs = run_shards(pkg, E, w, B, R, NAME[prec], True, g=g)
    assert abs(got["loss"] - rs["loss"]) <= 1e-6 * abs(rs["loss"]), (got["loss"], rs["loss"])
    assert trel(got["dE"], rs["dE"]) <= 2e-5, trel(got["dE"], rs["dE"])
    assert abs(got["dw"] - rs["dw"]) <= 1e-4 * max(1.0, abs(rs["dw"])), (got["dw"], rs["dw"])


# ------------------------------------------------------------------ rejected inputs leave no trace
def snapshot(ts):
    return [t.clone() for t in ts]


def unchanged(before, ts):
    """Bit-for-bit equality (NaN canaries included)."""
    return all(torch.equal(a.reshape(-1).view(torch.uint8), t.reshape(-1).view(torch.uint8))
               for a, t in zip(before, ts))


# (id, overrides of the call, expected code); base: N = 1024, M = 6, D = 256, 2 ranks, softmax, TF32
STEP_REJECTS = [
    ("one_rank", dict(n_ranks=1), SHAPE),
    ("nine_ranks", dict(n_ranks=9), SHAPE),
    ("n_local_times_ranks_not_n_total", dict(n_local=256), SHAPE),
    ("owner_rows_not_a_whole_tile", dict(N=1600, M=4, R=8), UNSUPPORTED),      # n_local = 200 on the TF32 path
    ("contrast", dict(variant=CONTRAST), UNSUPPORTED),
    ("simt_precision", dict(precision=FP32), UNSUPPORTED),
    ("misaligned_owner", dict(misalign=True), ARGUMENT),
    ("misaligned_owner_hyb", dict(misalign=True, hybrid=1), ARGUMENT),        # the conversion launch comes first
    ("misaligned_owner_split", dict(misalign=True, precision=FP32_SPLIT), ARGUMENT),   # ... the forward kernel
    ("null_owner", dict(null_owner=True), ARGUMENT),
]


@pytest.mark.parametrize("case,over,code", STEP_REJECTS, ids=[c[0] for c in STEP_REJECTS])
def test_step_rows_peers_rejects_without_a_trace(pkg, case, over, code):
    h = pkg.lib()
    N, M, D, R = over.get("N", 1024), over.get("M", 6), over.get("D", 256), over.get("R", 2)
    nl = N // R
    n_local, n_ranks = over.get("n_local", nl), over.get("n_ranks", R)
    variant, prec = over.get("variant", SOFTMAX), over.get("precision", TF32)
    U = nl * M
    if case == "owner_rows_not_a_whole_tile":
        assert h.ge2e_b200_path(nl, N, M, D, SOFTMAX, TF32) == 1 and nl % 128 != 0
    hyb_mode = over.get("hybrid", 0)
    assert hybrid_selected(h, nl, N, M, D, hyb_mode) == (hyb_mode == 1)
    h.ge2e_b200_debug_hybrid(hyb_mode)
    try:
        nb = max(h.ge2e_b200_workspace_bytes(nl, N, M, D, SOFTMAX, TF32), 256)
        gen = torch.Generator(device=DEV).manual_seed(7)
        f32 = dict(dtype=torch.float32, device=DEV)
        nan = float("nan")
        e_hat = torch.randn((U, D), generator=gen, **f32)
        c_hat = torch.randn((N, D), generator=gen, **f32)
        cos_diag = torch.rand(U, generator=gen, **f32)
        wt, bt, gt = (torch.tensor(v, **f32) for v in (W, B, 1.0))
        outs = [torch.full((U,), nan, **f32) for _ in range(3)]            # row_stat, row_aux, row_scale
        kstar = torch.full((U,), -7, dtype=torch.int32, device=DEV)
        accum = torch.full((4,), nan, **f32)
        dE_hat = torch.full((U, D), nan, **f32)
        d_buf = torch.full((n_ranks * (nl + 1) + 1, D), nan, **f32)       # owners' rows between NaN canaries
        owner = [d_buf[1 + r * (nl + 1):].data_ptr() for r in range(n_ranks)]
        if over.get("misalign"):
            owner[-1] += 4
        if over.get("null_owner"):
            owner[-1] = None
        ws = torch.zeros(nb, dtype=torch.uint8, device=DEV)
        everything = [e_hat, c_hat, cos_diag, wt, bt, gt, *outs, kstar, accum, dE_hat, d_buf, ws]
        torch.cuda.synchronize()
        before = snapshot(everything)
        n0 = h.ge2e_b200_launch_count()
        rc = h.ge2e_b200_step_rows_peers(e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(), n_local, N, 0, M, D,
                                         wt.data_ptr(), bt.data_ptr(), EPS, variant, prec, gt.data_ptr(),
                                         outs[0].data_ptr(), kstar.data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(),
                                         accum.data_ptr(), dE_hat.data_ptr(), ptrs(owner), n_ranks, ws.data_ptr(), nb,
                                         torch.cuda.current_stream().cuda_stream)
        launched = h.ge2e_b200_launch_count() - n0
        torch.cuda.synchronize()
    finally:
        h.ge2e_b200_debug_hybrid(0)
    assert rc == code, (rc, h.ge2e_b200_strerror(rc).decode())
    assert launched == 0, f"a refused call launched {launched} kernel(s)"
    assert unchanged(before, everything), "a refused call wrote into a buffer"


PUBLISH_REJECTS = [
    ("n_floats_not_a_float4_multiple", dict(n_floats=6), SHAPE),
    ("nine_destinations", dict(n_dst=9), SHAPE),
    ("multicast_with_two_destinations", dict(multicast=1, n_dst=2), SHAPE),
    ("misaligned_destination", dict(misalign=True), ARGUMENT),
]


@pytest.mark.parametrize("case,over,code", PUBLISH_REJECTS, ids=[c[0] for c in PUBLISH_REJECTS])
def test_peer_publish_rejects_without_a_trace(pkg, case, over, code):
    h = pkg.lib()
    n, slots = 1024, 9
    f32 = dict(dtype=torch.float32, device=DEV)
    src = torch.randn(n, generator=torch.Generator(device=DEV).manual_seed(3), **f32)
    dst = torch.full((slots, n + 4), float("nan"), **f32)          # 4 canary floats behind every destination
    zero = torch.full((n,), float("nan"), **f32)                    # the clear must not happen either
    n_dst, multicast, n_floats = over.get("n_dst", 2), over.get("multicast", 0), over.get("n_floats", n)
    dsts = [dst[i].data_ptr() for i in range(n_dst)]
    if over.get("misalign"):
        dsts[-1] += 4
    torch.cuda.synchronize()
    before = snapshot([src, dst, zero])
    n0 = h.ge2e_b200_launch_count()
    rc = h.ge2e_b200_peer_publish(src.data_ptr(), ptrs(dsts), n_dst, multicast, n_floats, zero.data_ptr(), n,
                                  torch.cuda.current_stream().cuda_stream)
    launched = h.ge2e_b200_launch_count() - n0
    torch.cuda.synchronize()
    assert rc == code, (rc, h.ge2e_b200_strerror(rc).decode())
    assert launched == 0
    assert unchanged(before, [src, dst, zero])


# ------------------------------------------------------------------ the reduce-scatter path: contrast, half E, g != 1
@pytest.mark.parametrize("N,M,D,R,g", [(64, 10, 256, 2, 1.0), (96, 5, 64, 3, 1.0), (64, 10, 256, 2, -1.5)])
@pytest.mark.parametrize("one_launch", [False, True])
def test_contrast_shards_simt_vs_oracle(pkg, N, M, D, R, g, one_launch):
    """Contrast on the SIMT kernels (path 0) with spk_offset > 0; finalize gets no row_scale."""
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, CONTRAST, FP32) == 0
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + R, kind="clustered"), device=DEV)
    ref = orct.forward_backward(E, W, B, EPS, "contrast", g=g)
    got = run_shards(pkg, E, W, B, R, "fp32", one_launch, variant=CONTRAST, g=g)
    check_dev(got, ref, N * M, FP32_TOL)


@pytest.mark.parametrize("one_launch", [False, True])
def test_contrast_shards_tc_forward_on_robust_rows(pkg, one_launch):
    """Contrast at config 3 on 8 shards: the TF32 tensor-core forward, then the SIMT gather backward.  dE is
    compared on the speakers TF32 rounding cannot touch (see test_cfg3_contrast_tf32_gradients_on_robust_rows)."""
    N, M, D, R = 1024, 10, 256, 8
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, CONTRAST, TF32) == 1
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=4, kind="random"), device=DEV)
    ref = orct.forward_backward(E, W, B, EPS, "contrast")
    got = run_shards(pkg, E, W, B, R, "tf32", one_launch, variant=CONTRAST)
    assert abs(got["loss"] - ref["loss"]) <= TF32_TOL * abs(ref["loss"])
    ok = robust_speakers(E, W)
    err = trel(got["dE"][ok], ref["dE"][ok].float())
    assert err <= TF32_TOL, err
    assert abs(got["dw"] - ref["dw"]) <= 2e-2 * max(1.0, abs(ref["dw"]))


# one rounding of dE to the embedding type, on top of the precision's class
HALF_ROUNDING = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}


@pytest.mark.parametrize("N,M,D,R,precision,path,g", [
    (512, 4, 256, 4, "fp32", 0, 1.0), (512, 4, 256, 4, "fp32_split", 2, 1.0),
    (1024, 10, 256, 8, "tf32", 1, 1.0), (1024, 10, 256, 8, "tf32", 1, -1.5),
])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("one_launch", [False, True])
def test_half_embedding_shards_vs_oracle(pkg, N, M, D, R, precision, path, g, dtype, one_launch):
    """bfloat16 / float16 E through prep_typed and bwd_finalize_typed on every shard; the oracle runs on the
    widened values."""
    from speaker_embedding_ge2e_loss_b200 import _lib
    assert pkg.lib().ge2e_b200_path(N // R, N, M, D, SOFTMAX, _lib.PRECISIONS[precision]) == path
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=N + R + 1, kind="clustered"), device=DEV).to(dtype)
    ref = orct.forward_backward(E, W, B, EPS, "softmax", g=g)
    got = run_shards(pkg, E, W, B, R, precision, one_launch, g=g)
    assert got["dE"].dtype == dtype
    tol = TF32_TOL if path == 1 else FP32_TOL
    assert abs(got["loss"] - ref["loss"]) <= tol * max(1.0, abs(ref["loss"])), (got["loss"], ref["loss"])
    r = trel(got["dE"].reshape(-1), ref["dE"].reshape(-1))
    assert r <= tol + HALF_ROUNDING[dtype], r
    assert abs(got["dw"] - ref["dw"]) <= tol * max(1.0, abs(ref["dw"])), (got["dw"], ref["dw"])
    assert abs(got["db"] - ref["db"]) <= 1e-5 * N * M, (got["db"], ref["db"])
