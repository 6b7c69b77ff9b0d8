"""What bf16 embeddings cost the loss step, against the two fp32 ways of running the same step.

    python scripts/half_io_cost.py --out DIR [--workload cfg3] [--precision tf32] [--steps 20] [--rounds 7]

Three CUDA graphs of ``--steps`` steps each, captured over the same rotating batches (more than the 126 MB L2
together, so every step reads its E from HBM), replayed alternately ``--rounds`` times in one process:

  bf16        GE2EPlan(dtype=torch.bfloat16) on bf16 E: prep reads E at half width, finalize writes bf16 dE
  workaround  what a bf16 model has to do without it: E.float() (a cast kernel and an fp32 copy of E), the fp32
              plan, then dE cast back to bf16 (a second cast kernel)
  fp32        the fp32 plan on fp32 E (the fp32 model's step: the reference point of bench.py)

It prints (and writes to DIR/half_io_cost.json) the median time per step of each, the GPU's name and power limit
read in the same run, and the largest difference between the bf16 plan's dE and the workaround's, in bf16 ulps
(the contract: the same fp32 numbers, rounded once to bf16, so 0 expected).
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


def ordered_bits(x: torch.Tensor) -> torch.Tensor:
    """bf16 bit patterns mapped to integers that are consecutive for consecutive bf16 values."""
    b = x.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(b < 0, -(b & 0x7FFF), b)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="tf32")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("half_io_cost.py needs a CUDA device")
    from speaker_embedding_ge2e_loss_b200 import GE2EPlan

    dev = torch.device("cuda:0")
    N, M, D = WORKLOADS[args.workload]
    U = N * M
    n_rot = max(2, int(np.ceil(1.5 * 126e6 / (U * D * 2))))       # bf16 batches alone exceed the L2
    E32 = [make_batch(N, M, D, seed=i).to(dev) for i in range(n_rot)]
    E16 = [e.to(torch.bfloat16) for e in E32]
    E32 = [e.float() for e in E16]           # the fp32 step sees the values the bf16 step sees
    w = torch.tensor(10.0, device=dev)
    b = torch.tensor(-5.0, device=dev)

    p16 = GE2EPlan(N, M, D, "softmax", args.precision, device=dev, dtype=torch.bfloat16)
    pwa = GE2EPlan(N, M, D, "softmax", args.precision, device=dev)
    p32 = GE2EPlan(N, M, D, "softmax", args.precision, device=dev)
    Ef = torch.empty((N, M, D), dtype=torch.float32, device=dev)        # the workaround's fp32 copy of E
    dE16_wa = torch.empty((N, M, D), dtype=torch.bfloat16, device=dev)

    def step_bf16(k):
        p16.step(E16[k % n_rot], w, b)

    def step_workaround(k):
        Ef.copy_(E16[k % n_rot])
        pwa.step(Ef, w, b)
        dE16_wa.copy_(pwa.dE)

    def step_fp32(k):
        p32.step(E32[k % n_rot], w, b)

    graphs = {"bf16": capture(step_bf16, args.steps), "workaround": capture(step_workaround, args.steps),
              "fp32": capture(step_fp32, args.steps)}
    for g in graphs.values():
        g.replay()
    torch.cuda.synchronize()
    times = {k: [] for k in graphs}
    for _ in range(args.rounds):
        for name, g in graphs.items():
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            e.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(e) * 1e3 / args.steps)

    # the last step of every graph ran on the same batch: compare the two bf16 gradients
    ulps = (ordered_bits(p16.dE) - ordered_bits(dE16_wa)).abs().max().item()
    res = {
        "workload": args.workload, "N": N, "M": M, "D": D, "precision": args.precision, "path": p16.path,
        "gpu": gpu_info(),
        "step_us_median": {k: float(np.median(v)) for k, v in times.items()},
        "step_us_rounds": {k: [round(x, 2) for x in v] for k, v in times.items()},
        "dE_bf16_vs_workaround_max_ulps": int(ulps),
        "loss": {"bf16": p16.loss.item(), "workaround": pwa.loss.item(), "fp32": p32.loss.item()},
        "how": (f"{args.steps} captured steps per graph over {n_rot} rotating batches ({n_rot * U * D * 2 / 1e6:.0f} MB "
                f"of bf16, {n_rot * U * D * 4 / 1e6:.0f} MB of fp32), the three graphs replayed alternately "
                f"{args.rounds} times; CUDA-event time per replay / steps, median over the rounds"),
    }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "half_io_cost.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    print("wrote", path)


if __name__ == "__main__":
    main()
