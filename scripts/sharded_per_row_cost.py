"""What the per-utterance losses cost one rank of the speaker-sharded peer-memory step, against the summed step.

    python scripts/sharded_per_row_cost.py --out DIR [--workloads cfg4x8,cfg3x8] [--steps 20] [--rounds 9]
                                           [--variant softmax|contrast]

cfg4x8 is config 4 (N = 8192, M = 16, D = 256) on 8 ranks (n_local = 1024), cfg3x8 config 3 (N = 1024, M = 10,
D = 256) on 8 ranks (n_local = 128), TF32.  One GPU plays one rank: every owner rank's dC_local lives on this device,
so the centroid pass's reduce-adds stay local (no NVLink traffic, no cross-rank barriers: those are not measured
here).  The rank's inputs (e_hat, c_hat_all, row statistics, dE_hat) rotate over enough sets to exceed the 126 MB L2,
every set with its own speaker offset, and every variant is a CUDA graph of ``--steps`` calls, replayed alternately
``--rounds`` times:

  sum       ge2e_b200_step_rows_peers: rows pass and centroid pass in one kernel
  none_fwd  ge2e_b200_fwd_rows with per_row, dE_hat and row_scale: the rows pass of reduction="none"
  none_bwd  ge2e_b200_bwd_rows_peers_per_row: the lone per-row centroid pass (+ the HYB conversion where it runs)
  none      none_fwd then none_bwd

--variant contrast times the contrast loss's peer-memory kernels against the reduce-scatter path's kernels instead
(both on the same rows pass, ge2e_b200_fwd_rows, which is the tensor-core contrast forward at these shapes):

  sum_peer  fwd_rows, then ge2e_b200_contrast_bwd_rows_peers adding into the owners' dC_local rows
  sum_rs    fwd_rows, then ge2e_b200_bwd_rows into a full-height dC_hat partial (the input of the reduce-scatter,
            which is not measured here, nor is the all-reduce of {loss, dw, db})
  none_peer / none_rs  the same with per_row and the per-row entry points (reduction="none")

It prints (and writes to DIR/sharded_per_row_cost.json, or sharded_contrast_cost.json) the median time per call, the
spread over the rounds, and the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from stage_profile import gpu_info  # noqa: E402

WORKLOADS = {"cfg4x8": (8192, 16, 256, 8), "cfg3x8": (1024, 10, 256, 8)}
L2_BYTES = 126 << 20


def check(h, rc, what):
    if rc != 0:
        raise RuntimeError(f"{what}: {h.ge2e_b200_strerror(rc).decode()}")


def capture(calls, steps):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        calls(0)                                 # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for k in range(steps):
            calls(k)
    return g


def measure(name, steps, rounds):
    import speaker_embedding_ge2e_loss_b200 as pkg
    h = pkg.lib()
    N, M, D, R = WORKLOADS[name]
    nl, U, prec = N // R, N // R * M, 1
    dev = torch.device("cuda")
    f32 = dict(dtype=torch.float32, device=dev)
    w, b, one = (torch.tensor(v, **f32) for v in (10.0, -5.0, 1.0))
    nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, 0, prec)
    per_set = 4 * (2 * U * D + N * D + 6 * U) + nb
    n_sets = max(2, -(-2 * L2_BYTES // per_set))
    owners_t = [torch.zeros((nl, D), **f32) for _ in range(R)]
    owners = (C.c_void_p * R)(*[t.data_ptr() for t in owners_t])
    gen = torch.Generator(device=dev).manual_seed(0)
    sets = []
    for k in range(n_sets):
        r = k % R
        E = torch.nn.functional.normalize(torch.randn((nl, M, D), generator=gen, **f32), dim=-1)
        c_all = torch.nn.functional.normalize(torch.randn((N, D), generator=gen, **f32), dim=-1)
        s = dict(r=r, E=E, c_all=c_all, e_hat=torch.empty((U, D), **f32), cos_diag=torch.empty(U, **f32),
                 accum=torch.empty(4, **f32), row_stat=torch.empty(U, **f32), row_aux=torch.empty(U, **f32),
                 kstar=torch.empty(U, dtype=torch.int32, device=dev), row_scale=torch.empty(U, **f32),
                 per=torch.empty(U, **f32), dE_hat=torch.empty((U, D), **f32),
                 g=torch.randn(U, generator=gen, **f32), ws=torch.zeros(nb, dtype=torch.uint8, device=dev))
        st = torch.cuda.current_stream().cuda_stream
        check(h, h.ge2e_b200_prep(E.data_ptr(), nl, M, D, prec, s["e_hat"].data_ptr(), c_all[r * nl:].data_ptr(),
                                  s["cos_diag"].data_ptr(), s["accum"].data_ptr(), st), "prep")
        sets.append(s)
    torch.cuda.synchronize()

    def fwd(k):
        s = sets[k % n_sets]
        check(h, h.ge2e_b200_fwd_rows(s["e_hat"].data_ptr(), s["c_all"].data_ptr(), s["cos_diag"].data_ptr(), nl, N,
                                      s["r"] * nl, M, D, w.data_ptr(), b.data_ptr(), 1e-6, 0, prec,
                                      s["row_stat"].data_ptr(), s["kstar"].data_ptr(), s["row_aux"].data_ptr(),
                                      s["accum"].data_ptr(), s["per"].data_ptr(), None, s["dE_hat"].data_ptr(),
                                      s["row_scale"].data_ptr(), s["ws"].data_ptr(), nb,
                                      torch.cuda.current_stream().cuda_stream), "fwd_rows")

    def bwd(k):
        s = sets[k % n_sets]
        check(h, h.ge2e_b200_bwd_rows_peers_per_row(
            s["e_hat"].data_ptr(), s["c_all"].data_ptr(), s["cos_diag"].data_ptr(), s["row_stat"].data_ptr(),
            s["row_aux"].data_ptr(), s["row_scale"].data_ptr(), nl, N, s["r"] * nl, M, D, w.data_ptr(), b.data_ptr(),
            1e-6, 0, prec, s["g"].data_ptr(), s["dE_hat"].data_ptr(), s["accum"].data_ptr() + 4, owners, R,
            s["ws"].data_ptr(), nb, torch.cuda.current_stream().cuda_stream), "bwd_rows_peers_per_row")

    def summed(k):
        s = sets[k % n_sets]
        check(h, h.ge2e_b200_step_rows_peers(
            s["e_hat"].data_ptr(), s["c_all"].data_ptr(), s["cos_diag"].data_ptr(), nl, N, s["r"] * nl, M, D,
            w.data_ptr(), b.data_ptr(), 1e-6, 0, prec, one.data_ptr(), s["row_stat"].data_ptr(), s["kstar"].data_ptr(),
            s["row_aux"].data_ptr(), s["row_scale"].data_ptr(), s["accum"].data_ptr(), s["dE_hat"].data_ptr(), owners,
            R, s["ws"].data_ptr(), nb, torch.cuda.current_stream().cuda_stream), "step_rows_peers")

    for k in range(n_sets):
        fwd(k)                                  # every set's row statistics exist before the backward runs alone
    torch.cuda.synchronize()
    variants = {"sum": summed, "none_fwd": fwd, "none_bwd": bwd, "none": lambda k: (fwd(k), bwd(k))}
    graphs = {v: capture(f, steps) for v, f in variants.items()}
    times = {v: [] for v in variants}
    for _ in range(rounds):
        for v, g in graphs.items():
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            g.replay()
            t1.record()
            t1.synchronize()
            times[v].append(t0.elapsed_time(t1) * 1e3 / steps)
    out = {"workload": name, "N": N, "M": M, "D": D, "ranks": R, "n_local": nl, "input_sets": n_sets,
           "input_bytes": n_sets * per_set, "steps_per_graph": steps, "rounds": rounds}
    for v, ts in times.items():
        out[v] = dict(median_us=float(np.median(ts)), min_us=float(np.min(ts)), max_us=float(np.max(ts)))
    return out


def measure_contrast(name, steps, rounds):
    import speaker_embedding_ge2e_loss_b200 as pkg
    h = pkg.lib()
    N, M, D, R = WORKLOADS[name]
    nl, U, prec, CONTRAST = N // R, N // R * M, 1, 1
    dev = torch.device("cuda")
    f32 = dict(dtype=torch.float32, device=dev)
    w, b, one = (torch.tensor(v, **f32) for v in (10.0, -5.0, 1.0))
    nb = h.ge2e_b200_workspace_bytes(nl, N, M, D, CONTRAST, prec)
    per_set = 4 * (2 * U * D + N * D + 6 * U) + nb
    n_sets = max(2, -(-2 * L2_BYTES // per_set))
    owners_t = [torch.zeros((nl, D), **f32) for _ in range(R)]
    owners = (C.c_void_p * R)(*[t.data_ptr() for t in owners_t])
    dC_partial = torch.empty((N, D), **f32)
    gen = torch.Generator(device=dev).manual_seed(0)
    sets = []
    for k in range(n_sets):
        r = k % R
        E = torch.nn.functional.normalize(torch.randn((nl, M, D), generator=gen, **f32), dim=-1)
        c_all = torch.nn.functional.normalize(torch.randn((N, D), generator=gen, **f32), dim=-1)
        s = dict(r=r, E=E, c_all=c_all, e_hat=torch.empty((U, D), **f32), cos_diag=torch.empty(U, **f32),
                 accum=torch.empty(4, **f32), row_stat=torch.empty(U, **f32), row_aux=torch.empty(U, **f32),
                 kstar=torch.empty(U, dtype=torch.int32, device=dev), per=torch.empty(U, **f32),
                 dE_hat=torch.empty((U, D), **f32), g=torch.randn(U, generator=gen, **f32),
                 ws=torch.zeros(max(nb, 1), dtype=torch.uint8, device=dev))
        st = torch.cuda.current_stream().cuda_stream
        check(h, h.ge2e_b200_prep(E.data_ptr(), nl, M, D, prec, s["e_hat"].data_ptr(), c_all[r * nl:].data_ptr(),
                                  s["cos_diag"].data_ptr(), s["accum"].data_ptr(), st), "prep")
        sets.append(s)
    torch.cuda.synchronize()

    def fwd(k, per_row):
        s = sets[k % n_sets]
        check(h, h.ge2e_b200_fwd_rows(s["e_hat"].data_ptr(), s["c_all"].data_ptr(), s["cos_diag"].data_ptr(), nl, N,
                                      s["r"] * nl, M, D, w.data_ptr(), b.data_ptr(), 1e-6, CONTRAST, prec,
                                      s["row_stat"].data_ptr(), s["kstar"].data_ptr(), s["row_aux"].data_ptr(),
                                      s["accum"].data_ptr(), s["per"].data_ptr() if per_row else None, None, None,
                                      None, s["ws"].data_ptr() if nb else None, nb,
                                      torch.cuda.current_stream().cuda_stream), "fwd_rows")

    def bwd_peer(k, per_row):
        s = sets[k % n_sets]
        fn = h.ge2e_b200_contrast_bwd_rows_peers_per_row if per_row else h.ge2e_b200_contrast_bwd_rows_peers
        check(h, fn(s["e_hat"].data_ptr(), s["c_all"].data_ptr(), s["cos_diag"].data_ptr(), s["row_stat"].data_ptr(),
                    s["kstar"].data_ptr(), nl, N, s["r"] * nl, M, D, w.data_ptr(), b.data_ptr(), 1e-6, prec,
                    (s["g"] if per_row else one).data_ptr(), s["dE_hat"].data_ptr(), s["accum"].data_ptr() + 4, owners,
                    R, torch.cuda.current_stream().cuda_stream), "contrast_bwd_rows_peers")

    def bwd_rs(k, per_row):
        s = sets[k % n_sets]
        fn = h.ge2e_b200_bwd_rows_per_row if per_row else h.ge2e_b200_bwd_rows
        check(h, fn(s["e_hat"].data_ptr(), s["c_all"].data_ptr(), s["cos_diag"].data_ptr(), s["row_stat"].data_ptr(),
                    s["kstar"].data_ptr(), s["row_aux"].data_ptr(), None, nl, N, s["r"] * nl, M, D, w.data_ptr(),
                    b.data_ptr(), 1e-6, CONTRAST, prec, (s["g"] if per_row else one).data_ptr(),
                    s["dE_hat"].data_ptr(), dC_partial.data_ptr(), s["accum"].data_ptr() + 4,
                    s["ws"].data_ptr() if nb else None, nb, torch.cuda.current_stream().cuda_stream), "bwd_rows")

    variants = {"sum_peer": lambda k: (fwd(k, False), bwd_peer(k, False)),
                "sum_rs": lambda k: (fwd(k, False), bwd_rs(k, False)),
                "none_peer": lambda k: (fwd(k, True), bwd_peer(k, True)),
                "none_rs": lambda k: (fwd(k, True), bwd_rs(k, True))}
    graphs = {v: capture(f, steps) for v, f in variants.items()}
    times = {v: [] for v in variants}
    for _ in range(rounds):
        for v, g in graphs.items():
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            g.replay()
            t1.record()
            t1.synchronize()
            times[v].append(t0.elapsed_time(t1) * 1e3 / steps)
    out = {"workload": name, "variant": "contrast", "precision": "tf32",
           "path": h.ge2e_b200_path(nl, N, M, D, CONTRAST, prec), "N": N, "M": M, "D": D, "ranks": R, "n_local": nl,
           "input_sets": n_sets, "input_bytes": n_sets * per_set, "steps_per_graph": steps, "rounds": rounds}
    for v, ts in times.items():
        out[v] = dict(median_us=float(np.median(ts)), min_us=float(np.min(ts)), max_us=float(np.max(ts)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_sharded_per_row"))
    ap.add_argument("--workloads", default="cfg4x8,cfg3x8")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--variant", default="softmax", choices=["softmax", "contrast"])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sharded_per_row_cost.py needs a CUDA device")
    res = {"gpu": gpu_info(), "results": []}
    print(json.dumps(res["gpu"]))
    contrast = args.variant == "contrast"
    shown = ("sum_peer", "sum_rs", "none_peer", "none_rs") if contrast else ("sum", "none_fwd", "none_bwd", "none")
    for name in args.workloads.split(","):
        r = (measure_contrast if contrast else measure)(name, args.steps, args.rounds)
        res["results"].append(r)
        print(name, {v: round(r[v]["median_us"], 2) for v in shown},
              f"sets={r['input_sets']} ({r['input_bytes'] / 2**20:.0f} MiB)", flush=True)
    os.makedirs(args.out, exist_ok=True)
    fname = "sharded_contrast_cost.json" if contrast else "sharded_per_row_cost.json"
    with open(os.path.join(args.out, fname), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
