"""What reduction="none" costs a training step, against the summed loss, and what the per-row backward costs against
the scalar one.

    python scripts/per_row_cost.py --out DIR [--workloads cfg2,cfg3] [--precisions fp32,tf32] [--steps 20] [--rounds 9]

Per (workload, precision), four CUDA graphs of ``--steps`` steps each, captured over rotating batches (more than the
126 MB L2 together, so every step reads its inputs from HBM), replayed alternately ``--rounds`` times in one process:

  sum          loss = GE2ELoss(reduction="sum")(E); loss.backward(): the whole step in the forward call (the
               single-kernel step at cfg2, prep + step kernel + finalize at cfg3), the upstream gradient applied by
               one scaling launch in backward
  none         L = GE2ELoss(reduction="none")(E); L.backward(g), g[N, M] random: the staged pipeline (forward kernels,
               then the per-row backward kernels)
  bwd_scalar   ge2e_b200_backward_typed alone, on saved forwards (one per rotating batch)
  bwd_per_row  ge2e_b200_backward_per_row_typed alone, on the same saved forwards

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


def measure(pkg, ops, lib_codes, workload, precision, steps, rounds, dev):
    N, M, D = WORKLOADS[workload]
    U = N * M
    vcode, pcode = lib_codes(precision, N, M, D)
    n_rot = max(2, int(np.ceil(1.5 * 126e6 / (U * D * 4))))
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
        "bwd_per_row_over_scalar": med["bwd_per_row"] / med["bwd_scalar"],
        "how": (f"{steps} captured steps per graph over {n_rot} rotating batches ({n_rot * U * D * 4 / 1e6:.0f} MB of "
                f"fp32 E), the four graphs replayed alternately {rounds} times; CUDA-event time per replay / steps, "
                "median and range over the rounds"),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="cfg2,cfg3")
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
