"""Outputs of the SIMT prep / finalize kernels and of the single-kernel step on fixed seeded inputs, for comparing
two builds of the library bit for bit.

    python scripts/stage_bits.py --lib path/to/libge2e_b200.so --out A.npz     # one build per process
    python scripts/stage_bits.py --compare A.npz B.npz      # A against B, degenerate speakers apart

Stages: ge2e_b200_prep_typed and ge2e_b200_bwd_finalize_typed on every body shape (register kernels: D = 128 / 256,
M <= 16; warp kernels: D = 256, M = 20 / 32 and D = 512; generic kernels: D = 100 / 192, an E at an 8-byte offset
(generic for fp32 only: the half types stay 8-byte aligned there), finalize at M = 40 (prep takes the warp kernel
at any M)), each E dtype, dE in fp32 and in E's type, every prep precision the body writes, both variants, with and
without row_scale, and an odd speaker count.  Finalize gets random dE_hat, dC_hat, cos_diag, row_aux and row_scale,
so its output depends on nothing but its inputs.  Speakers 0..4 of every case are degenerate (a zero row, rows of
norm 0.5 and 1.0 delta, a zero centroid, a zero leave-one-out centroid); --compare reports them apart.

Step: ge2e_b200_forward_backward_typed at cfg1, cfg2, N = 128 and one unaligned width (the single kernel's slow
path).  Its dE is assembled with L2 reduce-adds and is not deterministic: compare two runs of the same build for
the spread to set beside the difference between two builds.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

DELTA = 1e-8
DT = {"float32": 0, "bfloat16": 1, "float16": 2}
# (name, N, M, D, byte offset of E): the body the shape selects is named first
SHAPES = [("reg", 64, 2, 128, 0), ("reg", 64, 10, 128, 0), ("reg", 64, 16, 128, 0),
          ("reg", 64, 2, 256, 0), ("reg", 64, 10, 256, 0), ("reg", 64, 16, 256, 0), ("reg_odd", 7, 10, 256, 0),
          ("warp", 64, 20, 256, 0), ("warp", 64, 32, 256, 0), ("warp", 64, 10, 512, 0),
          ("generic", 64, 10, 100, 0), ("generic", 64, 10, 192, 0), ("generic_off8", 64, 10, 256, 8),
          ("generic", 32, 40, 256, 0)]
STEP_SHAPES = [("cfg1", 4, 8, 256), ("cfg2", 64, 10, 256), ("n128", 128, 10, 256), ("slow_d100", 16, 5, 100)]


def embeddings(N, M, D, seed):
    """Clustered rows with speakers 0..4 degenerate (as tests/test_gpu_edges.py builds them)."""
    rng = np.random.default_rng(seed)
    E = (rng.standard_normal((N, 1, D)) + 0.6 * rng.standard_normal((N, M, D))).astype(np.float32)
    deg = np.zeros(N, dtype=bool)
    if N < 5:
        return E, deg
    E[0, 1] = 0.0                                             # zero row (M = 2: zero leave-one-out of row 0)
    for j, s in ((1, 0.5), (2, 1.0)):                         # rows at and below the clamp
        E[j, 0] = (E[j, 0].astype(np.float64) * (s * DELTA / np.linalg.norm(E[j, 0].astype(np.float64)))).astype(np.float32)
    p = E[3, 0].copy()
    E[3] = 0.0
    E[3, 0], E[3, 1] = p, -p                                  # zero centroid
    if M >= 3:
        f = E[4, M - 1].copy()
        E[4] = 0.0
        E[4, 0], E[4, 1], E[4, M - 1] = p, -p, f              # zero leave-one-out centroid of the last row
    deg[:5] = True
    return E, deg


def run(libpath, out):
    import torch
    from speaker_embedding_ge2e_loss_b200 import _lib

    h = C.CDLL(os.path.abspath(libpath))
    for name, (res, args) in _lib.PROTOTYPES.items():
        fn = getattr(h, name)
        fn.restype, fn.argtypes = res, args
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    res = {}

    def put(key, t):
        res[key] = t.detach().float().cpu().numpy() if t.dtype != torch.int32 else t.cpu().numpy()

    def f32(*shape):
        return torch.full(shape, float("nan"), dtype=torch.float32, device=dev)

    w = torch.tensor(10.0, device=dev)
    b = torch.tensor(-5.0, device=dev)
    g = torch.tensor(0.75, device=dev)
    eps = 1e-6
    for si, (kind, N, M, D, off) in enumerate(SHAPES):
        E_np, deg = embeddings(N, M, D, seed=100 + si)
        U = N * M
        rng = np.random.default_rng(200 + si)
        dE_hat = torch.tensor(rng.standard_normal((U, D)).astype(np.float32) * 0.1, device=dev)
        dC_hat = torch.tensor(rng.standard_normal((N, D)).astype(np.float32) * 0.1, device=dev)
        cos_rand = torch.tensor(rng.uniform(-1, 1, U).astype(np.float32), device=dev)
        row_aux = torch.tensor(rng.uniform(0, 1, U).astype(np.float32), device=dev)
        row_scale = torch.tensor(rng.uniform(0.5, 2, U).astype(np.float32), device=dev)
        row_stat = torch.tensor(rng.uniform(0, 3, U).astype(np.float32), device=dev)
        for dname, dcode in DT.items():
            tdt = getattr(torch, dname)
            size = torch.tensor([], dtype=tdt).element_size()
            buf = torch.zeros(off // size + U * D + 8, dtype=tdt, device=dev)
            E = buf[off // size: off // size + U * D].view(U, D)
            E.copy_(torch.tensor(E_np.reshape(U, D), device=dev).to(tdt))
            case = f"{kind}_N{N}_M{M}_D{D}_{dname}"
            res[case + "/deg"] = np.repeat(deg, M)
            for prec in range(4):
                e_hat, c_hat, cos_diag, accum = f32(U, D), f32(N, D), f32(U), f32(4)
                rc = h.ge2e_b200_prep_typed(E.data_ptr(), dcode, None, N, M, D, prec, e_hat.data_ptr(),
                                            c_hat.data_ptr(), cos_diag.data_ptr(), accum.data_ptr(), st)
                torch.cuda.synchronize()
                res[f"{case}/prep{prec}/rc"] = np.array(rc)
                if rc == 0:
                    if prec >= 2:    # fp16 planes in the bytes of the fp32 rows: compare the bits
                        put(f"{case}/prep{prec}/e_hat", e_hat.view(torch.int32))
                        put(f"{case}/prep{prec}/c_hat", c_hat.view(torch.int32))
                    else:
                        put(f"{case}/prep{prec}/e_hat", e_hat)
                        put(f"{case}/prep{prec}/c_hat", c_hat)
                    put(f"{case}/prep{prec}/cos_diag", cos_diag)
            for ddname in sorted({"float32", dname}):
                for variant in (0, 1):
                    for rs in (False, True):
                        dE = torch.full((U, D), float("nan"), dtype=getattr(torch, ddname), device=dev)
                        rc = h.ge2e_b200_bwd_finalize_typed(
                            E.data_ptr(), dcode, None, dE_hat.data_ptr(), dC_hat.data_ptr(), cos_rand.data_ptr(),
                            row_stat.data_ptr(), row_aux.data_ptr(), row_scale.data_ptr() if rs else None, N, M, D,
                            w.data_ptr(), b.data_ptr(), eps, variant, g.data_ptr(), dE.data_ptr(), DT[ddname], st)
                        torch.cuda.synchronize()
                        key = f"{case}/fin_de{ddname}_v{variant}_rs{int(rs)}"
                        res[key + "/rc"] = np.array(rc)
                        if rc == 0:
                            put(key + "/dE", dE)
    for si, (name, N, M, D) in enumerate(STEP_SHAPES):
        E_np, deg = embeddings(N, M, D, seed=300 + si)
        U = N * M
        E = torch.tensor(E_np.reshape(U, D), device=dev)
        for variant in (0, 1):
            case = f"step_{name}_v{variant}"
            res[case + "/deg"] = np.repeat(deg, M)
            res[case + "/launches"] = np.array(h.ge2e_b200_step_launches(N, M, D, variant, 0))
            wsb = h.ge2e_b200_step_workspace_bytes(N, M, D, variant, 0)
            ws = torch.zeros(wsb, dtype=torch.uint8, device=dev)
            e_hat, c_hat, cos_diag, row_stat, row_aux, row_scale = f32(U, D), f32(N, D), f32(U), f32(U), f32(U), f32(U)
            row_kstar = torch.zeros(U, dtype=torch.int32, device=dev)
            accum, dE_hat, dC_hat, dE = f32(4), f32(U, D), f32(N, D), f32(U, D)
            rc = h.ge2e_b200_forward_backward_typed(
                E.data_ptr(), 0, None, N, M, D, w.data_ptr(), b.data_ptr(), eps, variant, 0, g.data_ptr(),
                e_hat.data_ptr(), c_hat.data_ptr(), cos_diag.data_ptr(), row_stat.data_ptr(), row_kstar.data_ptr(),
                row_aux.data_ptr(), row_scale.data_ptr(), accum.data_ptr(), dE_hat.data_ptr(), dC_hat.data_ptr(),
                dE.data_ptr(), 0, ws.data_ptr(), wsb, st)
            torch.cuda.synchronize()
            res[case + "/rc"] = np.array(rc)
            for k, t in (("e_hat", e_hat), ("c_hat", c_hat), ("cos_diag", cos_diag), ("dE", dE), ("accum", accum[:3])):
                put(f"{case}/{k}", t)
    np.savez_compressed(out, **res)
    print(f"{out}: {len(res)} arrays")


def diff(a, b, mask=None):
    """(bitwise equal, max |a - b|, max |a - b| / max |a|) over the rows of mask (None: all rows)."""
    if mask is not None:
        a, b = a[mask], b[mask]
    if a.size == 0:
        return True, 0.0, 0.0
    if a.dtype == np.int32:
        return bool(np.array_equal(a, b)), float(np.count_nonzero(a != b)), 0.0
    eq = bool(np.array_equal(a.view(np.uint32), b.view(np.uint32)))
    with np.errstate(invalid="ignore"):     # entries a kernel does not write stay NaN in both
        d = float(np.nanmax(np.abs(a.astype(np.float64) - b.astype(np.float64))))
    return eq, d, d / max(float(np.nanmax(np.abs(a))), 1e-30)


def compare(pa, pb):
    """One line per (body, stage, output, dE type): arrays compared, how many differ on the ordinary rows and on the
    degenerate speakers, and the largest max |a - b| / max |a| of each."""
    A, B = np.load(pa), np.load(pb)
    assert sorted(A.files) == sorted(B.files), "different case lists"
    groups = {}
    for k in sorted(A.files):
        if k.endswith("/rc") or k.endswith("/launches"):
            if int(A[k]) != int(B[k]):
                print(f"RETURN CODE MISMATCH {k}: {int(A[k])} vs {int(B[k])}")
            continue
        if k.endswith("/deg"):
            continue
        case, *sub = k.split("/")
        stage = "step" if case.startswith("step") else ("prep" if sub[0].startswith("prep") else "finalize")
        half_de = "fin_defloat16" in k or "fin_debfloat16" in k
        g = groups.setdefault((case.split("_N")[0].split("_v")[0], stage, sub[-1], "half" if half_de else "fp32"),
                              [0, 0, 0.0, 0, 0.0])
        deg = A[case + "/deg"]
        a, b = A[k], B[k]
        if a.shape[0] == deg.shape[0]:        # per-row arrays; c_hat and accum are not
            parts = ((1, diff(a, b, ~deg)), (3, diff(a, b, deg)))
        else:
            parts = ((1, diff(a, b)),)
        g[0] += 1
        for i, (eq, _, rel) in parts:
            if not eq:
                g[i] += 1
                g[i + 1] = max(g[i + 1], rel)
    print(f"{'body':12s} {'stage':8s} {'output':8s} {'dE':4s} {'arrays':>6s} | {'ordinary rows: differ':>21s} "
          f"{'max rel':>8s} | {'degenerate: differ':>18s} {'max rel':>8s}")
    for (body, stage, out, de), g in sorted(groups.items()):
        print(f"{body:12s} {stage:8s} {out:8s} {de:4s} {g[0]:6d} | {g[1]:21d} {g[2]:8.1e} | {g[3]:18d} {g[4]:8.1e}")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib")
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
    else:
        run(args.lib, args.out)
