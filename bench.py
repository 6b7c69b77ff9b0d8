#!/usr/bin/env python
"""GE2E loss fwd+bwd benchmark (BASELINE.json metric: utterances/s at N=1024, M=10, D=256).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg1|cfg2|cfg3|cfg4] [--precision tf32|fp32] [--variant softmax|contrast]
                    [--dump-outputs DIR]

One "step" = one GE2E forward + backward (grads to E, w, b) over one synthetic batch.
  value  device-resident inputs, the C-ABI calls of K consecutive steps captured in ONE CUDA graph
         (GE2EPlan.capture).  The inputs ROTATE over a set of batches larger than the 126 MB L2 (every step
         reads its batch from HBM); a replay of the K steps is bracketed by ONE pair of CUDA events on the
         launching stream; the reported time is the MEDIAN of 7 such replays (all listed in `replays_ms`).
  e2e    the same metric with the batch in pinned HOST memory: H2D copy of E and D2H read of loss / dw / db
         inside the timed region, through the public API (GE2EHostFeed, and the GE2ELoss module serially
         and double-buffered; the fastest is the headline, all three are listed with the API they use).
  roofline      the dominant kernel (the tensor-core step kernel: forward rows + both gradient
                contractions) priced IN SITU: every CTA stamps %globaltimer at its start and end
                (ge2e_b200_debug_stamps), the longest per-CTA (end - start) in the last step of a replay is the
                kernel's duration inside the running graph; algorithmic flops 6 U N D.
  fp32_path     cfg3 through the default precision of GE2ELoss(hp) ("fp32": fp32-class results; at this shape the
                tensor cores with operands split into two fp16 planes), same timing; the SIMT FMA kernels beside it.
  cpu_baseline  the reference's own GE2ELoss (baseline/_ref, unmodified) where its O(N^2 M D) expansion fits
                the host (cfg1, cfg2), else the torch-CPU port of it (oracle/ge2e_ref_port.py) on a bounded
                row sample of the same batch; all host threads.
N=1 runs cfg3 (the config the metric is quoted on).  N>1 runs cfg4 (N=8192, M=16) speaker-sharded over the
ranks (strong scaling: total work fixed); every rank checks its shard of the result against the single-GPU
plan on the same batch (parity_check, non-zero exit on failure) and rank 0 times cfg4 unsharded on its own
GPU so the line carries its own 1-GPU denominator (scaling_efficiency_same_workload).
--dump-outputs DIR writes what the K-th (last) timed step returned to its caller -- loss, dw, db and dE, float32 --
as DIR/<name>.npy (a sampled dE comes with its row indices, dE_rows.npy).  The batches are seeded and w = 10, b = -5, so the same arguments give the same inputs and two
builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    "cfg1": (4, 8, 256),
    "cfg2": (64, 10, 256),
    "cfg3": (1024, 10, 256),
    "cfg4": (8192, 16, 256),
}
METRIC = "GE2E fwd+bwd utterances/s"
UNIT = "utterances/s"
L2_FLUSH_BYTES = 256 << 20


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def ncu_traffic(kernel):
    """dram__bytes_read + dram__bytes_write per launch of `kernel`, from the committed ncu capture."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)["dram_bytes_per_launch"].get(kernel)
    except Exception:
        return None


def make_batch(N, M, D, seed=0):
    """Unit-scale random embeddings (SURVEY.md 8(d)): randn rows, L2-normalised, fp32."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N * M, D, generator=g)
    return (x / x.norm(dim=1, keepdim=True)).reshape(N, M, D).contiguous()


DUMP_BYTES = 64 << 20


def dump_row_ids(U, D):
    """Utterance rows of dE that --dump-outputs writes: all U when they fit 64 MB (less 1 MB kept for the
    scalars and the row indices), else a fixed seeded sample (numpy default_rng(0)), sorted.  cfg4's dE is 134 MB."""
    cap = (DUMP_BYTES - (1 << 20)) // (4 * D)
    if U <= cap:
        return np.arange(U)
    return np.sort(np.random.default_rng(0).choice(U, cap, replace=False))


def write_outputs(out_dir, outputs, N, M, D):
    """outputs: name -> float32 host array, dE as the [rows, D] rows of dump_row_ids.  Writes out_dir/<name>.npy:
    dE as [N, M, D] when it holds every row, else its rows plus their indices into [N * M, D] as dE_rows.npy
    (float64, exact).  Returns what the JSON line records."""
    rows = outputs["dE"].shape[0]
    if rows == N * M:
        outputs = dict(outputs, dE=outputs["dE"].reshape(N, M, D))
    else:
        outputs = dict(outputs, dE_rows=dump_row_ids(N * M, D).astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": os.path.abspath(out_dir), "shapes": {k: list(a.shape) for k, a in outputs.items()},
            "dE_rows": "all" if rows == N * M else
                       f"{rows} of {N * M} utterance rows of dE as [N * M, D], indices in dE_rows.npy (dump_row_ids)"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz, self._stop_evt = [], set(), None, threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # NVML missing: report it, do not fail the bench
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.02)

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "nvml unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- CPU reference arm
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def real_reference_class():
    """The reference's own GE2ELoss from baseline/_ref (scripts/install_reference.py), or None."""
    if not os.path.isfile(os.path.join(REF_DIR, "embedding_model_GE2E", "s3_loss_function_GE2E.py")):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        from embedding_model_GE2E.s3_loss_function_GE2E import GE2ELoss as RefLoss
        from utils.dict_to_dot import GetDictWithDotNotation
    except Exception:
        return None
    hp = GetDictWithDotNotation({"general": {"device": torch.device("cpu"), "small_err": 1e-6}})
    return lambda: RefLoss(hp)


def cpu_reference_sample(N, M, D, seed, target_rows):
    """Time the reference on the host cores: its own class on the whole batch where the O(N^2 M D)
    expansion fits (kind "reference"), else the port of it on a bounded row sample (kind "port").
    Returns (utt/s, dict)."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    U = N * M
    make = real_reference_class() if (target_rows >= U and U * N * D * 4 <= 2 << 30) else None
    if make is not None:
        crit = make()
        E = make_batch(N, M, D, seed).requires_grad_(True)
        best = None
        for it in range(3):
            E.grad = crit.w.grad = crit.b.grad = None
            t0 = time.perf_counter()
            loss = crit(E)
            loss.backward()
            dt = time.perf_counter() - t0
            best = dt if best is None or it > 0 and dt < best else best      # iteration 0 warms the allocator
        return U / best, dict(cores=threads, rows=U, seconds=best, kind="reference", loss=float(loss.detach()))
    from oracle import ge2e_ref_port as port
    E = make_batch(N, M, D, seed).numpy()
    rows = None if target_rows >= U else list(range(0, U, max(1, U // target_rows)))[:target_rows]
    sec, n_rows, _ = port.time_fwd_bwd(E, rows=rows, iters=1, warmup=0, threads=threads)
    return n_rows / sec, dict(cores=threads, rows=n_rows, seconds=sec, kind="port")


def config_of(wl, N, M, D, variant):
    """The `config` object: identical keys and values in both arms (the driver compares them)."""
    return {"workload": f"{wl}: N={N} M={M} D={D} {variant} GE2E fwd+bwd", "N": N, "M": M, "D": D, "variant": variant}


def cpu_sample_text(info, N, M):
    U = N * M
    if info["kind"] == "reference":
        return (f"the whole batch ({U} utterances), best of 2 timed iterations after 1 warm-up, {info['seconds']:.3f} s "
                f"each: the reference's own GE2ELoss (baseline/_ref/embedding_model_GE2E/s3_loss_function_GE2E.py, "
                f"unmodified) forward + backward on the host")
    return (f"{info['rows']} of {U} utterance rows against all {N} centroids, 1 iteration, {info['seconds']:.2f} s "
            f"(torch-CPU port of the reference's expanded algorithm, bit-checked against the real class; the full "
            f"batch needs {4 * U * N * 256 / 1e9:.0f} GB per expanded tensor and does not fit host RAM)")


def sample_rows_for(N, M, D):
    # ~1e9 expanded fp32 elements per tensor keeps host RSS < ~10 GB and the run in seconds
    return max(8, min(N * M, int(2.7e8 // (N * D))))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload or ("cfg3" if args.gpus == 1 else "cfg4")
    N, M, D = WORKLOADS[wl]
    # bound the whole run to a couple of minutes: ~5.5 ms of host time per row at cfg3
    rows = max(8, min(sample_rows_for(N, M, D), sample_rows_for(N, M, D) * 20 // max(1, args.steps + args.warmup)))
    vals, info = [], None
    for it in range(args.warmup + args.steps):
        v, info = cpu_reference_sample(N, M, D, seed=it, target_rows=rows)
        if it >= args.warmup:
            vals.append((v, info["seconds"]))
    value = float(np.median([v for v, _ in vals]))
    ms = float(np.median([s for _, s in vals])) * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic unit-norm random embeddings",
        "config": config_of(wl, N, M, D, args.variant),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                         "sample": cpu_sample_text(info, N, M) + " (per step)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- our arm
def timed_steps(fn, steps, warmup, flush_buf, pre=None):
    """fn() enqueues one step on the current stream.  Returns per-step milliseconds (device time)."""
    for _ in range(warmup):
        if pre:
            pre()
        flush_buf.fill_(1.0)
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        if pre:
            pre()
        flush_buf.fill_(1.0)                      # evict the 126 MB L2 between timed iterations
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def timed_back_to_back(plan, batches, w, b, steps, warmup, reps=7):
    """EXACTLY `steps` steps, rotating over `batches`, captured as ONE CUDA graph (the steps are
    stream-ordered exactly as a training loop would enqueue them).  The graph is replayed untimed
    until at least `warmup` steps have run (the first replay of a graph also pays its upload), then
    `reps` times, each inside one CUDA-event pair.  Returns (median ms per step, [ms per step of each replay])."""
    g = plan.capture(batches, w, b, steps=steps)
    for _ in range(max(1, -(-warmup // steps))):
        g.replay()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        e.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(e) / steps)
    return float(np.median(out)), out


def step_kernel_in_situ(plan, batches, w, b, steps, warmup, reps=11, all_out=None):
    """Duration of the tensor-core step kernel INSIDE the running graph: every CTA of the kernel stamps
    %globaltimer at its start and end (production kernel, two stores per CTA); after a replay the buffer
    holds the stamps of the replay's last step.  Returns the median over `reps` replays in microseconds,
    or None when the plan does not run the step kernel."""
    from speaker_embedding_ge2e_loss_b200 import lib
    h = lib()
    stamps = torch.zeros(2 * 512, dtype=torch.int64, device=batches[0].device)
    h.ge2e_b200_debug_stamps(stamps.data_ptr())
    try:
        g = plan.capture(batches, w, b, steps=steps)
        for _ in range(max(1, -(-warmup // steps))):
            g.replay()
        vals = []
        for _ in range(reps):
            stamps.zero_()
            g.replay()
            torch.cuda.synchronize()
            st = stamps.cpu().numpy().reshape(-1, 2)
            st = st[(st[:, 0] > 0) & (st[:, 1] > 0)]
            if len(st) == 0:
                return None
            # the longest per-CTA span (every CTA starts at the same event, the end of its predecessor grid): robust
            # against %globaltimer offsets between SMs, which max(end) - min(start) across CTAs is not (seen on some
            # boxes of the pool: cross-CTA spans LONGER than the whole step)
            vals.append(float((st[:, 1] - st[:, 0]).max()) / 1e3)
    finally:
        h.ge2e_b200_debug_stamps(None)
    if all_out is not None:
        all_out.extend(round(v, 2) for v in vals)
    return float(np.median(vals))


def stage_times(plan, E, w, b, flush_buf, reps=20):
    """CUDA-event time of each C-ABI stage (prep | step_rows | bwd_finalize) alone, L2 flushed before each."""
    from speaker_embedding_ge2e_loss_b200 import lib
    h = lib()
    N, M, D = plan.N, plan.M, plan.D
    s = torch.cuda.current_stream().cuda_stream
    ws = plan._ws.data_ptr() if plan._ws_bytes else None
    acc = plan._accum.data_ptr()
    scaled = plan.path in (1, 2, 3) and plan.variant == 0
    calls = {
        "prep": lambda: h.ge2e_b200_prep(E.data_ptr(), N, M, D, plan.precision, plan.e_hat.data_ptr(),
                                         plan.c_hat.data_ptr(), plan.cos_diag.data_ptr(), acc, s),
        "step_rows": lambda: h.ge2e_b200_step_rows(plan.e_hat.data_ptr(), plan.c_hat.data_ptr(), plan.cos_diag.data_ptr(),
                                                   N, N, 0, M, D, w.data_ptr(), b.data_ptr(), plan.eps, plan.variant,
                                                   plan.precision, plan.grad_out.data_ptr(), plan.row_stat.data_ptr(),
                                                   plan.row_kstar.data_ptr(), plan.row_aux.data_ptr(),
                                                   plan.row_scale.data_ptr(), acc, plan.dE_hat.data_ptr(),
                                                   plan.dC_hat.data_ptr(), ws, plan._ws_bytes, s),
        "bwd_finalize": lambda: h.ge2e_b200_bwd_finalize(E.data_ptr(), plan.dE_hat.data_ptr(), plan.dC_hat.data_ptr(),
                                                         plan.cos_diag.data_ptr(), plan.row_stat.data_ptr(),
                                                         plan.row_aux.data_ptr(),
                                                         plan.row_scale.data_ptr() if scaled else None, N, M, D,
                                                         w.data_ptr(), b.data_ptr(), plan.eps, plan.variant,
                                                         plan.grad_out.data_ptr(), plan.dE.data_ptr(), s),
    }
    out = {}
    for name, fn in calls.items():
        def run():
            rc = fn()
            assert rc == 0, (name, rc)
        ms = timed_steps(run, reps, 3, flush_buf)
        out[name] = float(np.median(ms)) * 1e3      # microseconds
    return out


def wait_for_clocks(sampler_index, seconds=3.0):
    """Spin a small kernel until NVML reports the SM clock within 5 % of its maximum (or `seconds` pass): a
    GPU that idled during host-side set-up ramps its clocks only gradually under a copy-dominated load."""
    try:
        import pynvml
        pynvml.nvmlInit()
        hd = pynvml.nvmlDeviceGetHandleByIndex(sampler_index)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(hd, pynvml.NVML_CLOCK_SM)
    except Exception:
        return None
    x = torch.randn(4096, 4096, device="cuda")
    t0 = time.perf_counter()
    mhz = 0
    while time.perf_counter() - t0 < seconds:
        for _ in range(20):
            x = torch.mm(x, x).clamp_(-1, 1)
        torch.cuda.synchronize()
        mhz = pynvml.nvmlDeviceGetClockInfo(hd, pynvml.NVML_CLOCK_SM)
        if mhz >= 0.95 * mx:
            break
    return {"sm_mhz": mhz, "sm_max_mhz": mx, "waited_s": round(time.perf_counter() - t0, 3)}


def measure_tf32_peak():
    """cuBLAS TF32 8192^3 burst, measured the way MEASURED_PEAKS.json measures bf16."""
    a = torch.randn(8192, 8192, device="cuda")
    b = torch.randn(8192, 8192, device="cuda")
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    best = 1e9
    for _ in range(3):
        torch.matmul(a, b)
    torch.cuda.synchronize()
    for _ in range(10):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.matmul(a, b)
        e.record()
        torch.cuda.synchronize()
        best = min(best, s.elapsed_time(e))
    torch.backends.cuda.matmul.allow_tf32 = old
    del a, b
    return 2 * 8192 ** 3 / (best * 1e-3) / 1e12


def run_ours(args):
    import torch.distributed as dist
    from speaker_embedding_ge2e_loss_b200 import GE2ELoss, GE2EPlan, lib
    from speaker_embedding_ge2e_loss_b200.sharded import shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rc = lib().ge2e_b200_check_device()
    if rc != 0:
        raise SystemExit("ge2e_b200: " + lib().ge2e_b200_strerror(rc).decode())

    wl = args.workload or ("cfg3" if world == 1 else "cfg4")
    N, M, D = WORKLOADS[wl]
    U = N * M
    peaks = load_peaks()
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=dev)
    w = torch.tensor(10.0, device=dev)
    b = torch.tensor(-5.0, device=dev)
    sampler = ClockSampler(local_rank)
    launches_before = lib().ge2e_b200_launch_count()
    extra = {}

    if world == 1:
        # inputs larger than L2: rotate over enough batches that a step never finds its E in the L2
        n_rot = max(2, int(np.ceil(1.5 * 126e6 / (U * D * 4))))
        batches = [make_batch(N, M, D, seed=i).to(dev) for i in range(n_rot)]
        E = batches[0]
        plan = GE2EPlan(N, M, D, args.variant, args.precision, device=dev)
        sampler.start()
        ms_med, replays = timed_back_to_back(plan, batches, w, b, args.steps, args.warmup)
        ms = [ms_med] * args.steps
        clocks = sampler.finish()
        extra["replays_ms"] = [round(x, 6) for x in replays]
        if args.dump_outputs:
            # the plan's buffers hold the last timed step (batch (K - 1) % n_rot); later measurements reuse them
            ids = torch.from_numpy(dump_row_ids(U, D)).to(dev)
            outputs = {"loss": plan.loss.cpu().numpy(), "dw": plan.dw.cpu().numpy(), "db": plan.db.cpu().numpy(),
                       "dE": plan.dE.reshape(U, D)[ids].cpu().numpy()}
        g1 = plan.capture(E, w, b)
        launches = plan.launches_per_step * args.steps
        extra["ms_per_step_l2_flushed"] = float(np.median(timed_steps(g1.replay, args.steps, args.warmup, flush)))
        path = plan.path
        g1.replay()
        loss_val = plan.loss.item()

        # ---- e2e: public module API, host-resident batch -------------------------------------
        crit = GE2ELoss(None, device=dev, variant=args.variant, precision=args.precision)
        E_host = make_batch(N, M, D, seed=0).pin_memory()
        res_host = torch.empty(3, dtype=torch.float32).pin_memory()

        def e2e_step():
            Ed = E_host.to(dev, non_blocking=True).requires_grad_(True)
            loss = crit(Ed)
            crit.w.grad = crit.b.grad = None
            loss.backward()
            res_host.copy_(torch.stack([loss.detach(), crit.w.grad, crit.b.grad]), non_blocking=True)

        e2e_ms = timed_steps(e2e_step, args.steps, args.warmup, flush)
        # host-side wall clock for the same loop (includes Python + autograd dispatch)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e_serial_t = max(float(np.mean(e2e_ms)), e2e_wall_ms)

        # the same K steps with the input feed double-buffered: the H2D copy of batch k+1 (copy stream)
        # runs under the fwd+bwd of batch k (compute stream); every step still copies its own batch in
        # from pinned host memory and its own loss / dw / db out, all inside the timed region
        copy_s = torch.cuda.Stream(device=dev)
        comp_s = torch.cuda.current_stream(dev)
        hosts = [make_batch(N, M, D, seed=i).pin_memory() for i in range(2)]
        bufs = [torch.empty((N, M, D), dtype=torch.float32, device=dev) for _ in range(2)]
        outs = [torch.empty(3, dtype=torch.float32).pin_memory() for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def pipelined(steps):
            used = [False, False]
            with torch.cuda.stream(copy_s):
                bufs[0].copy_(hosts[0], non_blocking=True)
                copied[0].record(copy_s)
            for k in range(steps):
                i, j = k % 2, (k + 1) % 2
                if k + 1 < steps:
                    with torch.cuda.stream(copy_s):
                        if used[j]:
                            copy_s.wait_event(consumed[j])
                        bufs[j].copy_(hosts[j], non_blocking=True)
                        copied[j].record(copy_s)
                comp_s.wait_event(copied[i])
                Ed = bufs[i].detach().requires_grad_(True)
                loss = crit(Ed)
                crit.w.grad = crit.b.grad = None
                loss.backward()
                outs[i].copy_(torch.stack([loss.detach(), crit.w.grad, crit.b.grad]), non_blocking=True)
                consumed[i].record(comp_s)
                used[i] = True

        pipelined(max(4, args.warmup))
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(comp_s)
        copy_s.wait_event(ev0)
        pipelined(args.steps)
        ev1.record(comp_s)
        torch.cuda.synchronize()
        e2e_pipe_wall = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e_pipe_dev = ev0.elapsed_time(ev1) / args.steps
        e2e_pipe_t = max(e2e_pipe_dev, e2e_pipe_wall)
        serial = {"value": U / (e2e_serial_t * 1e-3), "ms_per_step_device": float(np.mean(e2e_ms)),
                  "ms_per_step_wall": e2e_wall_ms,
                  "how": "copy, fwd+bwd and read-back serialised on one stream, L2 flushed between steps"}
        piped = {"value": U / (e2e_pipe_t * 1e-3), "ms_per_step_device": e2e_pipe_dev,
                 "ms_per_step_wall": e2e_pipe_wall,
                 "how": "H2D of batch k+1 on a copy stream under the fwd+bwd of batch k (double-buffered feed)"}
        # the host-fed plan (public API GE2EHostFeed): same double-buffered feed, each slot's step (stages +
        # the D2H read of loss/dw/db) is one CUDA graph, so the host issues a few stream calls per batch;
        # every step's result is read on the host (one step behind the submit)
        from speaker_embedding_ge2e_loss_b200 import GE2EHostFeed
        feed = GE2EHostFeed(N, M, D, w, b, args.variant, args.precision, device=dev)
        fhosts = [make_batch(N, M, D, seed=i).pin_memory() for i in range(3)]

        def fed(steps):
            prev, out = None, None
            for k in range(steps):
                t = feed.submit(fhosts[k % 3])
                if prev is not None:
                    out = feed.result(prev)
                prev = t
            return feed.result(prev)

        # warm-up: after the host-side set-up above the GPU has idled and its clocks ramp back only gradually
        # under this copy-dominated load (scripts/h2d_probe.py: 640 -> 195 us/step over ~250 steps on a fresh
        # feed).  Bring the SM clock back to its maximum with a compute kernel (NVML reading, not a rate
        # heuristic), then run a fixed 200 feed steps; steady state is what a training loop sees
        fed(max(4, args.warmup))
        fed_clock = wait_for_clocks(local_rank)
        fed(200)
        fed_warm = max(4, args.warmup) + 200
        torch.cuda.synchronize()
        fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        fe0.record(feed.copy_stream)
        fed_last = fed(args.steps)
        fe1.record(feed.compute_stream)
        torch.cuda.synchronize()
        fed_wall = (time.perf_counter() - t0) * 1e3 / args.steps
        fed_dev = fe0.elapsed_time(fe1) / args.steps
        fed_t = max(fed_dev, fed_wall)
        fedd = {"value": U / (fed_t * 1e-3), "ms_per_step_device": fed_dev, "ms_per_step_wall": fed_wall,
                "how": "GE2EHostFeed: H2D of batch k+1 on a copy stream under the graph-captured fwd+bwd+result read of "
                       "batch k; every step's loss/dw/db read on the host", "last_result": list(fed_last),
                "warmup_steps": fed_warm, "clock_before_warmup": fed_clock,
                "h2d_gbps": E_host.numel() * 4 / (fed_t * 1e-3) / 1e9}
        cands = {"host_fed_plan": fedd, "module_api_pipelined": piped, "module_api_serial": serial}
        bname = min(cands, key=lambda k: U / cands[k]["value"])
        best = cands[bname]
        apis = {"host_fed_plan": "GE2EHostFeed.submit / .result (graph-captured step per slot)",
                "module_api_pipelined": "GE2ELoss(hp)(E); loss.backward() (the call s4_train_embed_model.py:196-200 "
                                        "makes), batches double-buffered by the caller",
                "module_api_serial": "GE2ELoss(hp)(E); loss.backward() (the call s4_train_embed_model.py:196-200 makes)"}
        for k in cands:
            cands[k]["api"] = apis[k]
        e2e = {"value": best["value"], "unit": UNIT, "h2d_bytes_per_step": E_host.numel() * 4,
               "d2h_bytes_per_step": 12, "ms_per_step_device": best["ms_per_step_device"],
               "ms_per_step_wall": best["ms_per_step_wall"], "how": bname + ": " + best["how"], "api": apis[bname]}
        e2e.update({k: v for k, v in cands.items() if k != bname})

        # ---- roofline of the dominant kernel --------------------------------------------------
        st = stage_times(plan, E, w, b, flush)
        tf32_peak = measure_tf32_peak()
        extra["stage_us_alone_l2_flushed"] = st
        extra["tf32_cublas_tflops_measured_here"] = tf32_peak
        step_us = ms_med * 1e3
        flops = 6.0 * U * N * D
        kern_all = []
        kern_us = step_kernel_in_situ(plan, batches, w, b, max(10, args.steps), max(3, args.warmup),
                                      all_out=kern_all) if path in (1, 2, 3) else None
        if kern_us is not None and path == 2:
            dom, how = "tc_strip_kernel<STEP, split fp16 planes> (dE_hat pass + dC_hat pass; the rows were closed by the forward kernel before it)", \
                "in situ: the longest per-CTA (end - start) of the kernel's %globaltimer stamps in the last step of a graph replay (all CTAs start at the same event), median of 11 replays"
            extra["step_us_outside_the_step_kernel"] = step_us - kern_us
        elif kern_us is not None:
            dom, how = "tc_strip_kernel<STEP> (forward rows + dE_hat pass, grid barrier, dC_hat pass)", \
                "in situ: the longest per-CTA (end - start) of the kernel's %globaltimer stamps in the last step of a graph replay (all CTAs start at the same event), median of 11 replays"
            extra["step_us_outside_the_step_kernel"] = step_us - kern_us
        elif getattr(plan, "single_kernel", False):
            dom, kern_us, how = "small_step_kernel (whole fwd+bwd step)", step_us, "the step is this one kernel: step time"
        else:
            # SIMT pipeline (fp32 path, contrast backward): the rows kernels dominate; priced alone, L2 flushed
            dom, kern_us, how = "strip_kernel x3 (ge2e_b200_step_rows)", min(st["step_rows"], step_us), \
                "C-ABI stage timed alone between L2 flushes (CUDA events), capped by the step time"
        achieved = flops / (kern_us * 1e-6) / 1e12
        if path == 1:
            # a < 0.1 ms step is a burst; the multi-millisecond cfg4 step runs under the power cap
            key = "bf16_tflops" if wl != "cfg4" else "bf16_tflops_sustained"
            peak, peak_note = peaks[key] / 2, f"MEASURED_PEAKS {key}/2 (TF32 runs at half the bf16 rate), {peaks['source']}"
        elif path == 2:
            key = "bf16_tflops" if wl != "cfg4" else "bf16_tflops_sustained"
            peak, peak_note = peaks[key] / 3, (f"MEASURED_PEAKS {key}/3: an fp32-class product is three fp16 MMAs "
                                               f"(hi.hi + hi.lo + lo.hi) at the bf16 rate, {peaks['source']}")
        elif path == 3:
            key = "bf16_tflops" if wl != "cfg4" else "bf16_tflops_sustained"
            peak, peak_note = peaks[key], f"MEASURED_PEAKS {key} (fp16 operands run at the bf16 rate), {peaks['source']}"
        else:
            peak, peak_note = 148 * 128 * 2 * 1.965e9 / 1e12, "nominal fp32 FMA 148 SM x 128 lanes x 2 x 1.965 GHz (SIMT path; no measured entry)"
        roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": ncu_traffic("step") if (wl == "cfg3" and path == 1) else None,
                    "peak_source": peak_note,
                    "traffic_note": "DRAM bytes per launch from the committed ncu --set full capture (cold L2), see "
                                    "profiles/ncu_traffic.json; operands are L2-resident in situ",
                    "kernel_us": kern_us, "kernel_us_how": how, "kernel_us_replays": kern_all or None,
                    "algorithmic_flops": flops,
                    "issued_flops": 8.0 * U * N * D if path == 1 else (8.0 * U * N * D * 3 if path == 2 else None),
                    "note": ("algorithmic flops only (6 U N D: S, dE_hat, dC_hat); the second computation of S "
                             "for the dC_hat pass (another 2 U N D) is not credited") if path != 2 else
                            ("algorithmic flops only (6 U N D) against this ONE kernel, which issues 8 U N D x 3 fp16 MMAs; "
                             "the forward kernel in front of it (S once more, 2 U N D x 3) is outside kernel_us and inside "
                             "step_frac"),
                    "step_frac": (flops / (step_us * 1e-6) / 1e12) / peak}

        # ---- the default precision of the drop-in module on the same workload ----------------
        if wl == "cfg3" and args.precision == "tf32" and args.variant == "softmax":
            plan32 = GE2EPlan(N, M, D, args.variant, "fp32", device=dev)
            k32 = max(3, min(args.steps, 10))
            ms32, rep32 = timed_back_to_back(plan32, batches, w, b, k32, 3, reps=3)
            fma_peak = 148 * 128 * 2 * 1.965e9 / 1e12
            names = {0: "simt-fp32", 1: "tcgen05-tf32", 2: "tcgen05 split fp16 planes (3 MMAs per product)"}
            extra["fp32_path"] = {"ms_per_step": ms32, "value": U / (ms32 * 1e-3), "unit": UNIT, "steps": k32,
                                  "replays_ms": [round(x, 5) for x in rep32], "path": names[plan32.path],
                                  "launches_per_step": 4 if plan32.path == 2 else None,
                                  "frac_vs_fp32_fma_roof": (flops / (ms32 * 1e-3) / 1e12) / fma_peak,
                                  "frac_vs_tf32_roof_div3": (flops / (ms32 * 1e-3) / 1e12) / (peaks["bf16_tflops"] / 2 / 3),
                                  "frac_vs_f16_roof_div3": (flops / (ms32 * 1e-3) / 1e12) / (peaks["bf16_tflops"] / 3),
                                  "loss": float(plan32.loss.item()),
                                  "note": "GE2ELoss(hp) defaults to precision='fp32' (reference arithmetic, 1e-5 parity, "
                                          "tests/test_gpu_split.py): this line.  At this shape it runs on the tensor cores with "
                                          "every operand split into two fp16 planes (GE2E_FP32_SPLIT); precision='tf32' (or "
                                          "hp.general.ge2e_precision) selects the TF32 path of the headline, 'fp32_simt' the "
                                          "fp32 FMA kernels"}
            del plan32
            plan_simt = GE2EPlan(N, M, D, args.variant, "fp32_simt", device=dev)
            ms_s, _ = timed_back_to_back(plan_simt, batches, w, b, 3, 2, reps=3)
            extra["fp32_path"]["simt_fp32_ms_per_step"] = ms_s
            del plan_simt
    else:
        from speaker_embedding_ge2e_loss_b200.sharded import sharded_ge2e_loss
        off, n_local = shard_bounds(N, world, rank)
        E_full = make_batch(N, M, D, seed=0)
        E = E_full[off:off + n_local].contiguous().to(dev).requires_grad_(True)
        wp = w.clone().requires_grad_(True)
        bp = b.clone().requires_grad_(True)

        def step():
            E.grad = wp.grad = bp.grad = None
            loss = sharded_ge2e_loss(E, wp, bp, 1e-6, args.variant, args.precision)
            loss.backward()
            return loss

        dist.barrier()
        if os.environ.get("GE2E_BENCH_SHARDED_EAGER") == "1":
            sampler.start()
            ms = timed_steps(step, args.steps, args.warmup, flush, pre=dist.barrier)
            clocks = sampler.finish()
            t = torch.tensor([float(np.sum(ms))], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = [t.item() / args.steps] * args.steps
            sharded_how = "eager autograd path, CUDA events per step, L2 flushed, max over ranks"
        else:
            # the K steps (stages + NCCL collectives) captured as ONE CUDA graph over persistent buffers,
            # this rank's shard rotating over more batches than fit the L2; one warm replay, then one
            # timed replay between barriers; device time, max over ranks
            from speaker_embedding_ge2e_loss_b200 import ShardedGE2EPlan
            n_rot = max(2, int(np.ceil(1.5 * 126e6 / (n_local * M * D * 4))))
            shards = [make_batch(N, M, D, seed=i)[off:off + n_local].contiguous().to(dev) for i in range(n_rot)]
            shards[0] = E.detach()
            splan = ShardedGE2EPlan(n_local, N, off, M, D, args.variant, args.precision, device=dev)
            g = splan.capture(shards, w, b, steps=args.steps)
            for _ in range(max(1, -(-args.warmup // args.steps))):
                g.replay()
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            sampler.start()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            g.replay()
            ev1.record()
            torch.cuda.synchronize()
            clocks = sampler.finish()
            t = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = [t.item() / args.steps] * args.steps
            if args.dump_outputs:
                # loss / dw / db are global; every rank holds its speakers' rows of dE and sends rank 0 the sampled ones
                ids = dump_row_ids(U, D)
                lo = off * M
                mine = torch.from_numpy(ids[(ids >= lo) & (ids < lo + n_local * M)] - lo).to(dev)
                parts = [None] * world if rank == 0 else None
                dist.gather_object(splan.dE.reshape(-1, D)[mine].cpu().numpy(), parts, dst=0)
                if rank == 0:
                    outputs = {"loss": splan.loss.cpu().numpy(), "dw": splan.dw.cpu().numpy(),
                               "db": splan.db.cpu().numpy(), "dE": np.concatenate(parts)}
            splan.step(shards[0], w, b)                     # same batch as the checks below
            torch.cuda.synchronize()
            extra["sharded_loss_check"] = {"graph_plan": splan.loss.item()}
            # ---- parity: every rank runs the WHOLE batch through the single-GPU plan on its own GPU and
            # compares its shard of dE and the global loss / dw / db; the worst rank decides
            tol = 2e-3 if args.precision == "tf32" else 1e-5
            E1 = E_full.to(dev)
            plan1 = GE2EPlan(N, M, D, args.variant, args.precision, device=dev)
            plan1.step(E1, w, b)
            torch.cuda.synchronize()
            ref_dE = plan1.dE[off:off + n_local].double()
            errs = torch.tensor([
                ((splan.dE.double() - ref_dE).norm() / ref_dE.norm().clamp_min(1e-30)).item(),
                abs(splan.loss.item() - plan1.loss.item()) / max(1.0, abs(plan1.loss.item())),
                abs(splan.dw.item() - plan1.dw.item()) / max(1.0, abs(plan1.dw.item())),
                abs(splan.db.item() - plan1.db.item()) / (1e-5 * U / tol),       # db: absolute 1e-5 * U
            ], device=dev, dtype=torch.float64)
            dist.all_reduce(errs, op=dist.ReduceOp.MAX)
            parity = {"dE_rel": errs[0].item(), "loss": errs[1].item(), "dw": errs[2].item(),
                      "db_abs": errs[3].item() * (1e-5 * U / tol), "tol": tol, "ok": bool((errs <= tol).all().item()),
                      "against": "GE2EPlan on the whole batch on each rank's own GPU (max over ranks); the plan itself "
                                 "is checked against the float64 oracle at this size in tests/test_gpu_step.py"}
            extra["parity_check"] = parity
            del E1, plan1
            exchange = ("peer memory over NVLink (multicast publish of c_hat, step kernel reduce-adds dC_hat into the owner "
                        "rank, symmetric-memory barriers; no NCCL kernel in the step)" if splan.peer
                        else "NCCL all-gather / reduce-scatter / all-reduce")
            extra["exchange"] = {"peer_memory": bool(splan.peer), "multicast": bool(getattr(splan, "_mcast", 0)),
                                 "peer_error": splan.peer_error, "how": exchange}
            sharded_how = (f"K steps incl. the exchange steps ({exchange}) in one CUDA graph, shard rotating over {n_rot} "
                           f"batches ({n_rot * n_local * M * D * 4 / 1e6:.0f} MB), one event pair, max over ranks")
        launches = int(lib().ge2e_b200_launch_count() - launches_before)
        from speaker_embedding_ge2e_loss_b200 import _lib as _l
        vcode = 0 if args.variant == "softmax" else 1
        path = lib().ge2e_b200_path(n_local, N, M, D, vcode, _l.resolve_precision(args.precision, n_local, N, M, D, vcode))
        loss_val = step().item()
        e2e = None
        roofline = None
        if rank == 0:
            # host-resident e2e on the sharded path: each rank copies its shard in, reads the loss out
            pass

    if world > 1:
        # e2e for the sharded run: every rank H2D-copies its shard and reads back the global loss
        E_host = E_full[off:off + n_local].contiguous().pin_memory()
        res_host = torch.empty(1, dtype=torch.float32).pin_memory()

        def e2e_step():
            Ed = E_host.to(dev, non_blocking=True).requires_grad_(True)
            wp.grad = bp.grad = None
            loss = sharded_ge2e_loss(Ed, wp, bp, 1e-6, args.variant, args.precision)
            loss.backward()
            res_host.copy_(loss.detach().reshape(1), non_blocking=True)

        e2e_ms = timed_steps(e2e_step, args.steps, args.warmup, flush, pre=dist.barrier)
        t = torch.tensor([float(np.sum(e2e_ms))], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_t = t.item() / args.steps
        eager = {"value": U / (e2e_t * 1e-3), "ms_per_step": e2e_t,
                 "how": "eager sharded autograd path, copy + step + read-back serialised on one stream"}
        e2e = {"value": eager["value"], "unit": UNIT, "h2d_bytes_per_step": E_host.numel() * 4 * world,
               "d2h_bytes_per_step": 4 * world, "how": "module_api_eager: " + eager["how"]}
        if os.environ.get("GE2E_BENCH_SHARDED_EAGER") != "1":
            # host-fed sharded plan: every rank feeds its shard from pinned host memory (H2D of batch k+1 under
            # the graph-captured sharded step of batch k) and reads the global loss/dw/db of every step
            from speaker_embedding_ge2e_loss_b200 import ShardedGE2EHostFeed
            feed = ShardedGE2EHostFeed(n_local, N, off, M, D, w, b, args.variant, args.precision, device=dev)
            fhosts = [make_batch(N, M, D, seed=i)[off:off + n_local].contiguous().pin_memory() for i in range(3)]

            def fed(steps):
                prev = None
                for k in range(steps):
                    tk = feed.submit(fhosts[k % 3])
                    if prev is not None:
                        feed.result(prev)
                    prev = tk
                return feed.result(prev)

            def fed_timed(steps):                       # wall time between barriers, max over ranks
                torch.cuda.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                out = fed(steps)
                torch.cuda.synchronize()
                tt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                return tt.item(), out

            fed(max(4, args.warmup))
            last, fed_warm = None, max(4, args.warmup)
            for _ in range(10):                         # settle (decided on the all-reduced time: ranks stay in lockstep)
                cur, _ = fed_timed(20)
                fed_warm += 20
                if last is not None and abs(cur - last) <= 0.03 * last:
                    break
                last = cur
            fed_s, fed_last = fed_timed(args.steps)
            fed_t = fed_s * 1e3 / args.steps
            fedd = {"value": U / (fed_t * 1e-3), "ms_per_step": fed_t, "warmup_steps": fed_warm,
                    "last_result": list(fed_last),
                    "how": "ShardedGE2EHostFeed: per rank, H2D of shard k+1 on a copy stream under the graph-captured "
                           "sharded step (stages + NCCL) of shard k; every step's global loss/dw/db read on the host; "
                           "wall clock between barriers, max over ranks"}
            if fedd["value"] > e2e["value"]:
                e2e = {"value": fedd["value"], "unit": UNIT, "h2d_bytes_per_step": E_host.numel() * 4 * world,
                       "d2h_bytes_per_step": 12 * world, "ms_per_step": fed_t, "how": "host_fed_plan: " + fedd["how"],
                       "warmup_steps": fed_warm, "last_result": fedd["last_result"], "module_api_eager": eager}
            else:
                e2e["host_fed_plan"] = fedd
        # long steps: sustained rates.  TF32 = half the bf16 rate; an fp32-class product = three fp16 MMAs
        peak = (peaks["bf16_tflops_sustained"] / 2 if path == 1 else
                peaks["bf16_tflops_sustained"] / 3 if path == 2 else 148 * 128 * 2 * 1.965e9 / 1e12)
        ach = 6.0 * U * N * D / (ms[0] * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "whole sharded step, all ranks", "achieved": ach,
                    "peak": peak * world, "unit": "TFLOP/s", "frac": ach / (peak * world), "traffic": None,
                    "peak_source": "MEASURED_PEAKS bf16_tflops_sustained / 2 (TF32) or / 3 (split fp16 planes) per GPU "
                                   "(millisecond-long steps run under the power cap)"}
        if rank == 0:
            # 1-GPU denominator for strong scaling: the same cfg on this rank's GPU alone
            E1 = E_full.to(dev)
            plan1 = GE2EPlan(N, M, D, args.variant, args.precision, device=dev)
            g1 = plan1.capture(E1, w, b)
            ms1 = float(np.median(timed_steps(g1.replay, max(5, args.steps // 2), 3, flush)))
            extra["single_gpu_same_workload"] = {"value": U / (ms1 * 1e-3), "unit": UNIT, "ms_per_step": ms1}
            extra["scaling_efficiency_same_workload"] = ms1 / (world * ms[0])
            del E1, plan1, g1
        dist.barrier()

    if world > 1:
        g = splan = feed = shards = fhosts = step = e2e_step = fed = fed_timed = None   # drop the graphs that hold NCCL nodes
    if world > 1 and not extra.get("parity_check", {"ok": True})["ok"]:
        if rank == 0:
            print(json.dumps({"error": "sharded result does not match the single-GPU plan", **extra["parity_check"]}))
        _leave(world, code=3)
    if rank != 0:
        _leave(world)
        return

    ms_per_step = float(np.mean(ms))
    value = U / (ms_per_step * 1e-3)
    cpu_val, cpu_info = cpu_reference_sample(N, M, D, seed=0, target_rows=sample_rows_for(N, M, D)) \
        if world == 1 else (None, None)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
        "dtype": {1: "tf32", 2: "f16x2-split (fp32-class)", 3: "f16"}.get(path, "f32"),
        "data": "synthetic unit-norm random embeddings",
        "config": config_of(wl, N, M, D, args.variant),
        "run": {"precision": args.precision,
                "path": {1: "tcgen05-tf32", 2: "tcgen05 split fp16 planes", 3: "tcgen05 fp16 operands"}.get(path, "simt-fp32"),
                "parallelism": "replica" if world == 1 else f"speakers sharded x{world} (all-gather c_hat, reduce-scatter dC_hat)",
                "l2": (f"inputs larger than L2: the step rotates over {n_rot} batches ({n_rot * U * D * 4 / 1e6:.0f} MB), "
                       "no flush") if world == 1 else sharded_how,
                "timing": "median of 7 replays of the K steps captured as one CUDA graph, one CUDA-event pair per replay"
                if world == 1 else sharded_how},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "loss": loss_val,
    }
    if cpu_val is not None:
        line["cpu_baseline"] = {"value": cpu_val, "unit": UNIT, "cores": cpu_info["cores"], "kind": cpu_info["kind"],
                                "sample": cpu_sample_text(cpu_info, N, M)}
    if args.dump_outputs:
        line["outputs"] = write_outputs(args.dump_outputs, outputs, N, M, D)
    line.update(extra)
    print(json.dumps(line))
    _leave(world)


def _leave(world, code=0):
    """End a multi-rank run.  The instantiated CUDA graphs that hold NCCL collectives are destroyed FIRST
    (garbage-collect every plan / feed / graph object, synchronise); only then is the communicator torn down.
    Destroying it while such a graph was alive blocked both ranks in round 1.  The teardown runs under a
    watchdog: all results are out by now, so a communicator that still refuses to die within 20 s does not
    turn a finished measurement into a failure."""
    if world <= 1:
        if code:
            sys.exit(code)
        return
    import gc
    import torch.distributed as dist
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    gc.collect()
    torch.cuda.synchronize()
    killer = threading.Timer(20.0, lambda: os._exit(code))
    killer.daemon = True
    killer.start()
    try:
        dist.destroy_process_group()
    except Exception:
        pass
    killer.cancel()
    sys.stdout.flush()
    os._exit(code)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="tf32", choices=["tf32", "fp32", "fp32_simt", "fp32_split", "f16"])
    ap.add_argument("--variant", default="softmax", choices=["softmax", "contrast"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write loss, dw, db and dE of the last one as DIR/<name>.npy (float32; "
                         "dE rows sampled to keep the total under 64 MB, their indices in dE_rows.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or os.environ.get("GE2E_BENCH_SHARDED_EAGER") == "1"):
        ap.error("--dump-outputs writes the outputs of the CUDA-graph timed path of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
