"""Step time and in-situ kernel time of GE2EPlan (graph of K steps over rotating batches > L2).

    python scripts/step_probe.py [cfg3|cfg4|N,M,D] [--precision tf32|fp32] [--steps K] [--reps R] [--trace]

Prints one JSON line: ms per step (median of R replays), the step kernel's duration inside the running
graph (ge2e_b200_debug_stamps: per-CTA globaltimer start / end of the LAST step of a replay), and with
--trace a per-role timeline of the slowest cluster from the instrumented instantiation.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from speaker_embedding_ge2e_loss_b200 import GE2EPlan, lib  # noqa: E402

CFG = {"cfg1": (4, 8, 256), "cfg2": (64, 10, 256), "cfg3": (1024, 10, 256), "cfg4": (8192, 16, 256)}


def batch(N, M, D, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N * M, D, generator=g)
    return (x / x.norm(dim=1, keepdim=True)).reshape(N, M, D).contiguous().to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("shape", nargs="?", default="cfg3")
    ap.add_argument("--precision", default="tf32")
    ap.add_argument("--variant", default="softmax")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--trace", action="store_true")
    ap.add_argument("--fine", action="store_true", help="with --trace: one mark per ring stage in the MMA warp")
    ap.add_argument("--hybrid", type=int, default=0, help="ge2e_b200_debug_hybrid mode (-1 never, 0 default rule, 1 always)")
    a = ap.parse_args()
    N, M, D = CFG[a.shape] if a.shape in CFG else tuple(int(v) for v in a.shape.split(","))
    dev = torch.device("cuda:0")
    U = N * M
    n_rot = max(2, int(np.ceil(1.5 * 126e6 / (U * D * 4))))
    batches = [batch(N, M, D, i, dev) for i in range(n_rot)]
    w, b = torch.tensor(10.0, device=dev), torch.tensor(-5.0, device=dev)
    h = lib()
    h.ge2e_b200_debug_hybrid(a.hybrid)
    plan = GE2EPlan(N, M, D, a.variant, a.precision, device=dev)
    stamps = torch.zeros(2 * 148 * 2, dtype=torch.int64, device=dev)
    h.ge2e_b200_debug_stamps(stamps.data_ptr())
    g = plan.capture(batches, w, b, steps=a.steps)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    ms = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / a.steps)
    st = stamps.cpu().numpy().reshape(-1, 2)
    st = st[st[:, 0] > 0]
    out = {"shape": [N, M, D], "precision": a.precision, "path": plan.path, "launches_per_step": plan.launches_per_step,
           "ms_per_step_median": float(np.median(ms)), "ms_per_step_all": [round(x, 5) for x in ms],
           "utt_per_s": U / (float(np.median(ms)) * 1e-3)}
    if len(st):
        out["step_kernel_us_in_situ"] = float(st[:, 1].max() - st[:, 0].min()) / 1e3
        out["step_kernel_cta_us"] = {"min": float((st[:, 1] - st[:, 0]).min()) / 1e3,
                                     "max": float((st[:, 1] - st[:, 0]).max()) / 1e3, "ctas": int(len(st))}
        out["algorithmic_tflops_step_kernel"] = 6.0 * U * N * D / (out["step_kernel_us_in_situ"] * 1e-6) / 1e12
    out["algorithmic_tflops_step"] = 6.0 * U * N * D / (float(np.median(ms)) * 1e-3) / 1e12
    h.ge2e_b200_debug_stamps(None)
    print(json.dumps(out))
    if a.trace:
        ev = 64
        tr = torch.zeros(148 * 3 * ev, dtype=torch.int64, device=dev)
        h.ge2e_b200_debug_trace(tr.data_ptr(), 1 | (0x100 if a.fine else 0))
        plan.step(batches[0], w, b)
        torch.cuda.synchronize()
        h.ge2e_b200_debug_trace(None, -1)
        t = tr.cpu().numpy().reshape(148, 3, ev)
        # fixed slots of the epilogue record: [61] pass 1 done, [62] pass 2 begins, [63] ns waiting for row sums
        fixed = t[:, 2, ev - 3:].copy()
        t[:, 2, ev - 3:] = 0
        t0 = t[t > 0].min()
        ends = np.array([t[c][t[c] > 0].max() if (t[c] > 0).any() else 0 for c in range(148)])
        for c in (0, int(np.argmax(ends)), int(np.argmin(np.where(ends > 0, ends, ends.max())))):
            for role, name in enumerate(("tma", "mma", "epi")):
                v = t[c, role]
                v = v[v > 0]
                print(f"cta {c:3d} {name}: " + " ".join(f"{(x - t0) / 1e3:.1f}" for x in v))
        print("per CTA (us from kernel start): pass-1 done, pass-2 begins, total wait for pass-2 row sums")
        for c in range(148):
            p1, p2, wait = fixed[c]
            if p1 or p2 or wait:
                f = lambda x: f"{(x - t0) / 1e3:6.1f}" if x else "     -"
                print(f"cta {c:3d}: {f(p1)} {f(p2)} {wait / 1e3:6.2f}")


if __name__ == "__main__":
    main()
