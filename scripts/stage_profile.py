"""Per-kernel time of the fwd+bwd step inside the CUDA graph that bench.py times.

    python scripts/stage_profile.py --out DIR [--workload cfg3] [--precision tf32] [--variant softmax]
                                    [--dtype float32|bfloat16|float16] [--steps 20] [--replays 5]

The step is captured the way bench.py captures it: GE2EPlan.capture over batches rotated so that their
total exceeds the 126 MB L2 (every step reads its E from HBM).  First the graph is replayed with the
profiler off and timed with CUDA events (median ms per step over the replays).  Then one more series of
replays runs under torch.profiler with CUDA activities, and every kernel launch of it is attributed to
prep (prep_*kernel), finalize (finalize_*kernel) or the step between them (everything else the library
launches: the tensor-core kernels, or the SIMT rows kernels).  The kernels are launched with programmatic
dependent launch, so a kernel starts while its predecessor runs and waits inside: its duration overlaps the
predecessor's.  Each launch is therefore also given its exclusive time, end - max(start, end of the previous
kernel), which is what it adds to the step; the exclusive times of a step and the gaps between its kernels
add up to the step time.  The medians per kernel and per role go to DIR/stage_profile.json together with the
GPU's name and power limit, read in the same run.  ``--dtype`` is the element type of the embeddings (and of dE):
the plan is built with ``GE2EPlan(dtype=...)`` and the batches are converted once, before the capture.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import WORKLOADS, make_batch  # noqa: E402


def gpu_info():
    """Card name, power limit and maximum SM clock (a read-only nvidia-smi query)."""
    info = {"name": torch.cuda.get_device_name()}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                              "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        info.update(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as exc:  # noqa: BLE001 -- the numbers stand without it, marked as such
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def role(name):
    if "prep" in name and "kernel" in name:
        return "prep"
    if "finalize" in name:
        return "finalize"
    return "step"


def short(name):
    """Kernel name without return type, namespaces and parameter list; template arguments kept."""
    name = name.replace("(anonymous namespace)::", "").replace("ge2e::", "").removeprefix("void ")
    if name.endswith(")"):      # cut the parameter list: the '(' that matches the final ')'
        depth = 0
        for i in range(len(name) - 1, -1, -1):
            depth += {")": 1, "(": -1}.get(name[i], 0)
            if depth == 0:
                return name[:i]
    return name


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory (created)")
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="tf32")
    ap.add_argument("--variant", default="softmax", choices=["softmax", "contrast"])
    ap.add_argument("--dtype", default="float32", choices=["float32", "bfloat16", "float16"])
    ap.add_argument("--steps", type=int, default=20, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage_profile.py needs a CUDA device")
    from speaker_embedding_ge2e_loss_b200 import GE2EPlan

    dev = torch.device("cuda:0")
    N, M, D = WORKLOADS[args.workload]
    U = N * M
    dtype = getattr(torch, args.dtype)
    esize = torch.empty((), dtype=dtype).element_size()
    n_rot = max(2, int(np.ceil(1.5 * 126e6 / (U * D * esize))))
    batches = [make_batch(N, M, D, seed=i).to(dev, dtype) for i in range(n_rot)]
    w = torch.tensor(10.0, device=dev)
    b = torch.tensor(-5.0, device=dev)
    plan = GE2EPlan(N, M, D, args.variant, args.precision, device=dev, dtype=dtype)
    g = plan.capture(batches, w, b, steps=args.steps)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()

    step_ms = []
    for _ in range(args.replays):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        e.record()
        torch.cuda.synchronize()
        step_ms.append(a.elapsed_time(e) / args.steps)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.replays):
            g.replay()
        torch.cuda.synchronize()
    evs = sorted((ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA
                  and "memset" not in ev.name.lower() and "memcpy" not in ev.name.lower()),
                 key=lambda ev: ev.time_range.start)
    kernels = {}
    prev_end = None
    for ev in evs:
        t0, t1 = ev.time_range.start, ev.time_range.end
        excl = t1 - max(t0, prev_end) if prev_end is not None else None
        prev_end = t1 if prev_end is None else max(prev_end, t1)
        k = kernels.setdefault(ev.name, {"us": [], "excl": []})
        k["us"].append(t1 - t0)
        if excl is not None:
            k["excl"].append(max(0.0, excl))

    per_kernel = {}
    by_role = {"prep": [], "step": [], "finalize": []}
    excl_role = {"prep": [], "step": [], "finalize": []}
    for name, k in kernels.items():
        us, ex = k["us"], k["excl"] or [float("nan")]
        per_kernel[short(name)] = {"role": role(name), "launches": len(us), "median_us": float(np.median(us)),
                                   "min_us": float(np.min(us)), "max_us": float(np.max(us)),
                                   "median_exclusive_us": float(np.median(ex))}
        per_step = len(us) / (args.steps * args.replays)
        by_role[role(name)].append(float(np.median(us)) * per_step)
        excl_role[role(name)].append(float(np.median(ex)) * per_step)
    res = {
        "workload": args.workload, "N": N, "M": M, "D": D, "precision": args.precision, "variant": args.variant,
        "dtype": args.dtype, "path": plan.path, "gpu": gpu_info(),
        "step_us": float(np.median(step_ms)) * 1e3, "step_us_replays": [round(x * 1e3, 2) for x in step_ms],
        "kernel_us_per_step": {k: round(sum(v), 3) for k, v in by_role.items()},
        "exclusive_us_per_step": {k: round(sum(v), 3) for k, v in excl_role.items()},
        "kernels": per_kernel,
        "how": (f"GE2EPlan.capture of {args.steps} steps over {n_rot} rotating batches ({n_rot * U * D * esize / 1e6:.0f} MB, "
                f"more than the L2); step_us = median over {args.replays} replays of CUDA-event time / steps, profiler "
                f"off; kernel times from one torch.profiler run of {args.replays} more replays (CUDA activities), the "
                "median duration (and median exclusive time) of each kernel times its launches per step, summed "
                "per role"),
    }
    res["step_us_outside_the_kernels"] = res["step_us"] - sum(res["exclusive_us_per_step"].values())
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "stage_profile.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("workload", "precision", "variant", "dtype", "gpu", "step_us", "kernel_us_per_step",
                                          "exclusive_us_per_step", "step_us_outside_the_kernels")}))
    for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1]["median_us"] * kv[1]["launches"]):
        print(f"  {v['role']:9s} {v['median_us']:8.2f} us (exclusive {v['median_exclusive_us']:7.2f}) x {v['launches']:4d}  {k}")
    print("wrote", path)


if __name__ == "__main__":
    main()
