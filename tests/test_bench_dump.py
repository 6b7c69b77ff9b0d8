"""bench.py --dump-outputs: the files hold what the last timed step computed (checked against the float64
oracle on the batch that step read), and the dE row sample keeps every workload's dump within 64 MB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import ge2e_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_rows_fit_the_budget_and_are_fixed():
    for N, M, D in bench.WORKLOADS.values():
        ids = bench.dump_row_ids(N * M, D)
        assert ids.size * (D * 4 + 8) + 3 * 4 <= bench.DUMP_BYTES      # dE rows, their float64 indices, scalars
        assert ids[0] >= 0 and ids[-1] < N * M and np.all(np.diff(ids) > 0)
        np.testing.assert_array_equal(ids, bench.dump_row_ids(N * M, D))
    N, M, D = bench.WORKLOADS["cfg3"]
    assert bench.dump_row_ids(N * M, D).size == N * M          # the headline workload is written whole


def test_sampled_dump_writes_its_row_indices(tmp_path):
    N, M, D = bench.WORKLOADS["cfg4"]
    ids = bench.dump_row_ids(N * M, D)
    dE = np.random.default_rng(1).standard_normal((ids.size, D)).astype(np.float32)
    s = np.zeros((), np.float32)
    info = bench.write_outputs(tmp_path, {"loss": s, "dw": s, "db": s, "dE": dE}, N, M, D)
    rows = np.load(tmp_path / "dE_rows.npy")
    assert rows.dtype == np.float64 and np.array_equal(rows.astype(np.int64), ids)
    assert np.array_equal(np.load(tmp_path / "dE.npy"), dE) and info["shapes"]["dE_rows"] == [ids.size]
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= bench.DUMP_BYTES


@pytest.mark.gpu
@pytest.mark.parametrize("steps", [1, 3])
def test_bench_dumps_the_last_timed_step(tmp_path, steps):
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg2", "--precision", "fp32",
                        "--steps", str(steps), "--warmup", "3", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    N, M, D = bench.WORKLOADS["cfg2"]
    got = {k: np.load(out / f"{k}.npy") for k in ("loss", "dw", "db", "dE")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["dE"].shape == (N, M, D) and line["outputs"]["shapes"]["dE"] == [N, M, D]
    # step k of the timed graph reads batch seed k (cfg2 rotates over hundreds of batches): the last is steps - 1
    ref = orc.forward_backward(bench.make_batch(N, M, D, seed=steps - 1).numpy(), 10.0, -5.0, 1e-6, "softmax")
    assert abs(float(got["loss"]) - ref["loss"]) <= 1e-5 * abs(ref["loss"])
    assert abs(float(got["dw"]) - ref["dw"]) <= 1e-5 * max(1.0, abs(ref["dw"]))
    # db is the eps term alone (zero in exact arithmetic) and cancels in fp32 sums: bounded, as in test_gpu_parity;
    # loss, dw and dE are what pin the step
    assert abs(float(got["db"]) - ref["db"]) <= 1e-5 * N * M
    assert np.linalg.norm(got["dE"] - ref["dE"]) <= 1e-5 * np.linalg.norm(ref["dE"])
