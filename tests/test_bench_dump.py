"""bench.py --dump-outputs: what the timed path returned in its last step, written as .npy files within the size budget."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_budget_and_fixed_sample(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 4 * 1000)
    arrays = {"small": torch.arange(10, dtype=torch.float64).reshape(2, 5),
              "mid": torch.arange(300, dtype=torch.float32),
              "big": torch.arange(50_000, dtype=torch.float32).reshape(100, 500)}
    got = bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert sum(k for _, k in got.values()) <= 1000
    assert got["small"] == ((2, 5), 10) and got["mid"] == ((300,), 300) and got["big"][0] == (100, 500)
    for name in arrays:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), arrays["small"].float().numpy())
    big = np.load(tmp_path / "a" / "big.npy")                 # values of arange = the flat indices sampled
    k = got["big"][1]
    assert big.shape == (k,) and k < 50_000
    lo = np.arange(k) * 50_000 // k
    assert ((big >= lo) & (big < lo + 50_000 // k)).all()      # one element from each of k equal strides


@pytest.mark.gpu
def test_bench_dump_matches_oracle(tmp_path):
    """the dumped loss, outputs and gradients of a small run are those of the fp64 oracle on the same seeded inputs, and
    --steps sets the number of timed steps."""
    from parity_util import W, is_dead, oracle_step, relerr
    d = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "2", "--batch", "2", "--steps", "3",
                          "--warmup", "1", "--precision", "fp32", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    assert sum(f.stat().st_size for f in d.iterdir()) <= 64 << 20
    w = W.make_workload(2, 2)
    ref = oracle_step(w, 2)
    assert abs(float(np.load(d / "loss.npy")[0]) - ref["loss"]) <= 1e-5 * abs(ref["loss"])
    assert relerr(torch.from_numpy(np.load(d / "out.npy")), ref["out"]) <= 1e-5
    assert relerr(torch.from_numpy(np.load(d / "hidden.npy")), ref["hid"]) <= 1e-5
    n = 0
    for k, g in ref["grads"].items():
        if not is_dead(w.model, k):
            got = torch.from_numpy(np.load(d / f"grad.{k}.npy"))
            assert relerr(got, g) <= (1e-4 if k.endswith("_attention") else 1e-5), k
            n += 1
    assert n >= 10
