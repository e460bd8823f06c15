"""bench.py contract checks that do not need a GPU: the reference arm's code path (with CPU stand-ins for the CUDA-event
timer and the NVML clock sampler) and the shape of its JSON line."""
import contextlib
import json
import os
import sys
import time
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class _CpuTimer:
    def __init__(self, warmup, steps, on_start=None, on_stop=None):
        self.warmup, self.steps, self.count = warmup, steps, 0

    def step(self):
        self.count += 1
        if self.count == self.warmup:
            self.t0 = time.perf_counter()
        elif self.count == self.warmup + self.steps:
            self.t1 = time.perf_counter()

    def ms(self):
        return (self.t1 - self.t0) * 1e3


class _NoClocks:
    def __init__(self, index):
        pass

    def start(self):
        pass

    def stop(self):
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}


def test_reference_arm_runs_the_unmodified_reference(monkeypatch):
    import bench
    ref = bench.ensure_reference()
    if ref is None:
        pytest.skip("oracle/_ref not installed (build() installs it from a checkout of the reference)")
    monkeypatch.setattr(bench, "StepTimer", _CpuTimer)
    monkeypatch.setattr(bench, "ClockSampler", _NoClocks)
    monkeypatch.setattr(bench, "REF_SAMPLES_PER_NODE", 128)
    monkeypatch.setattr(bench, "NODES_PER_GPU", 3)
    import torch
    dtype = torch.get_default_dtype()
    try:
        with contextlib.redirect_stdout(sys.stderr):
            out = bench._reference_rank0(types.SimpleNamespace(gpus=1, warmup=3, steps=2, extras=False), ref, "fp64", 60.0)
    finally:
        torch.set_default_dtype(dtype)            # the stock runner switches the process to float64
        for m in [k for k in sys.modules if k.split(".")[0] in ("models", "optimizers", "problems", "utils")]:
            sys.modules.pop(m, None)
        if ref in sys.path:
            sys.path.remove(ref)
    line = json.loads(json.dumps(out))
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "impl"):
        assert key in line, key
    assert line["impl"] == "reference" and line["steps"] == 2 and line["dtype"] == "fp64" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0
    # both arms print the same config dict (the driver compares them)
    assert line["config"] == bench.headline_config(1)


def test_dump_outputs_writes_compact_rows_within_the_size_cap(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    from nn_distributed_training_b200.models import MNISTConvNet
    from nn_distributed_training_b200.parallel.arena import FlatLayout, NodeArena
    from nn_distributed_training_b200.parallel.context import DistContext

    arena = NodeArena(FlatLayout.from_module(MNISTConvNet(3, 5, 64)), 3, "cpu", torch.float64)
    arena.theta.normal_()
    pr = types.SimpleNamespace(arena=arena, gather_rows=lambda t: t,
                               fused=types.SimpleNamespace(loss_part=torch.rand(3, 2)))
    opt = types.SimpleNamespace(duals=arena.theta * 2)
    bench.dump_outputs(str(tmp_path / "full"), DistContext.single(), pr, opt)
    got = {n: np.load(tmp_path / "full" / f"{n}.npy") for n in ("theta", "duals", "losses")}
    np.testing.assert_array_equal(got["theta"], arena.compact(arena.theta).numpy())
    np.testing.assert_array_equal(got["duals"], 2 * got["theta"])
    np.testing.assert_array_equal(got["losses"], pr.fused.loss_part.sum(1).numpy())
    assert got["theta"].dtype == np.float64 and got["losses"].dtype == np.float32

    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 200_000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), DistContext.single(), pr, opt)
    small = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("theta", "duals", "losses")}
    assert sum(a.nbytes for a in small.values()) <= 200_000 and 0 < small["theta"].shape[1] < got["theta"].shape[1]
    np.testing.assert_array_equal(small["duals"], 2 * small["theta"])
    np.testing.assert_array_equal(small["theta"], np.load(tmp_path / "b" / "theta.npy"))      # the same sample every run


def test_reference_arm_caps_the_timed_region():
    import bench
    # 8 "GPUs" x 10 nodes at 4.65 ms per node-round: 1000 requested rounds would take 6 minutes
    n_nodes = bench.NODES_PER_GPU * 8
    k = min(1000, max(5, int(bench.REF_MAX_SECONDS / (bench.REF_SEC_PER_NODE_ROUND * n_nodes)) - 5))
    assert 100 < k < 1000 and k * bench.REF_SEC_PER_NODE_ROUND * n_nodes <= bench.REF_MAX_SECONDS
