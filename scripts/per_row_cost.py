"""What reduction="none" costs a training step, against the summed loss, and what the per-row backward costs against
the scalar one.

    python scripts/per_row_cost.py --out DIR [--workloads cfg2,cfg3,128x10x256] [--precisions fp32,tf32] [--steps 20]
                                   [--rounds 9]

A workload is a bench.py name or NxMxD.  Per (workload, precision), five CUDA graphs of ``--steps`` steps each,
captured over up to ``--steps`` rotating batches, replayed alternately ``--rounds`` times in one process.  At cfg3 the
batches together exceed the 126 MB L2, so every step reads its inputs from HBM; at the small workloads (cfg1, cfg2,
128x10x256) they fit in the L2 and the numbers are those of L2-resident inputs, as in a training loop at these sizes.


  sum          loss = GE2ELoss(reduction="sum")(E); loss.backward(): the whole step in the forward call (the
               single-kernel step at cfg2, prep + step kernel + finalize at cfg3), the upstream gradient applied by
               one scaling launch in backward
  none         L = GE2ELoss(reduction="none")(E); L.backward(g), g[N, M] random: the forward kernels, then the
               per-row backward kernels (on the single-kernel step's shapes one launch each, else the staged pipeline)
  bwd_scalar   ge2e_b200_backward_typed alone, on saved forwards (one per rotating batch)
  bwd_per_row  ge2e_b200_backward_per_row_typed alone, on the same saved forwards
  plan_none    GE2EPlan(reduction="none").step(E, w, b): the per-row forward and backward as bare C-ABI calls
               (grad_rows = g of the first batch); skipped on a build whose GE2EPlan has no reduction argument

It prints (and writes to DIR/per_row_cost.json) the median time per step of each, the spread over the rounds, and
the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import WORKLOADS, make_batch  # noqa: E402
from stage_profile import gpu_info  # noqa: E402


def capture(step, steps):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step(0)                                  # warm-up outside the capture (module load, lazy attributes)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for k in range(steps):
            step(k)
    return g


def shape_of(workload):
    if workload in WORKLOADS:
        return WORKLOADS[workload]
    N, M, D = (int(x) for x in workload.split("x"))
    return N, M, D


def measure(pkg, ops, lib_codes, workload, precision, steps, rounds, dev):
    N, M, D = shape_of(workload)
    U = N * M
    vcode, pcode = lib_codes(precision, N, M, D)
    n_rot = min(steps, max(2, int(np.ceil(1.5 * 126e6 / (U * D * 4)))))   # a graph uses `steps` batches at most
    Es = [make_batch(N, M, D, seed=i).to(dev).requires_grad_(True) for i in range(n_rot)]
    gen = torch.Generator().manual_seed(0)
    gs = [torch.randn(N, M, generator=gen).to(dev) for _ in range(n_rot)]
    crit_sum = pkg.GE2ELoss(None, device=dev, precision=precision)
    crit_none = pkg.GE2ELoss(None, device=dev, precision=precision, reduction="none")

    def step_sum(k):
        crit_sum(Es[k % n_rot]).backward()

    def step_none(k):
        crit_none(Es[k % n_rot]).backward(gs[k % n_rot])

    # saved forwards for the backward-only graphs: the tensor-core softmax paths prepare dE_hat / row_scale
    w, b = crit_none.w.detach(), crit_none.b.detach()
    saved = [ops._fwd_impl(E.detach(), w, b, crit_none.eps, vcode, pcode, per_row=True)
             for E in Es]
    one = torch.ones((), device=dev)

    def bwd(k, per_row):
        E = Es[k % n_rot].detach()
        _, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale = saved[k % n_rot]
        g = gs[k % n_rot] if per_row else one
        ops._bwd_impl(g, E, w, b, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, dE_hat, row_scale,
                      crit_none.eps, vcode, pcode, per_row=per_row)

    graphs = {"sum": capture(step_sum, steps), "none": capture(step_none, steps),
              "bwd_scalar": capture(lambda k: bwd(k, False), steps),
              "bwd_per_row": capture(lambda k: bwd(k, True), steps)}
    try:
        plan = pkg.GE2EPlan(N, M, D, precision=precision, device=dev, reduction="none")
    except TypeError:
        plan = None
    if plan is not None:
        plan.grad_rows.copy_(gs[0])
        wp, bp = w.clone(), b.clone()
        graphs["plan_none"] = plan.capture([E.detach() for E in Es], wp, bp, steps=steps)
        plan_launches = plan.launches_per_step
    for g in graphs.values():
        g.replay()
    torch.cuda.synchronize()
    times = {k: [] for k in graphs}
    for _ in range(rounds):
        for name, g in graphs.items():
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            e.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(e) * 1e3 / steps)
    med = {k: float(np.median(v)) for k, v in times.items()}
    return {
        "workload": workload, "N": N, "M": M, "D": D, "precision": precision,
        "path": crit_none.path_for(N, M, D),
        "step_us_median": med,
        "step_us_min_max": {k: [round(min(v), 2), round(max(v), 2)] for k, v in times.items()},
        "none_over_sum": med["none"] / med["sum"],
        "plan_none_over_sum": med["plan_none"] / med["sum"] if plan is not None else None,
        "plan_none_launches_per_step": plan_launches if plan is not None else None,
        "bwd_per_row_over_scalar": med["bwd_per_row"] / med["bwd_scalar"],
        "how": (f"{steps} captured steps per graph over {n_rot} rotating batches ({n_rot * U * D * 4 / 1e6:.0f} MB of "
                f"fp32 E), the graphs replayed alternately {rounds} times; CUDA-event time per replay / steps, "
                "median and range over the rounds"),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="cfg1,cfg2,128x10x256,cfg3")
    ap.add_argument("--precisions", default="fp32,tf32")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=9)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("per_row_cost.py needs a CUDA device")
    import speaker_embedding_ge2e_loss_b200 as pkg
    from speaker_embedding_ge2e_loss_b200 import _lib, ops

    def lib_codes(precision, N, M, D):
        v = _lib.VARIANTS["softmax"]
        return v, _lib.resolve_precision(precision, N, N, M, D, v)

    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "results": []}
    for wl in args.workloads.split(","):
        for prec in args.precisions.split(","):
            r = measure(pkg, ops, lib_codes, wl, prec, args.steps, args.rounds, dev)
            print(json.dumps(r), flush=True)
            res["results"].append(r)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "per_row_cost.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))
    print("wrote", path)


if __name__ == "__main__":
    main()
