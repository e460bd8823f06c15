"""GPU numerics of the fp64 density kernels (csrc/mlp_f64.cu) against float64 autograd.

Every comparison starts the fused problem and a ``backend="torch"`` twin from the same parameters.  Both compute in
float64, so they may differ only by summation order: ~1e-14 relative typically, ~4e-12 in the worst case for the
2e4-term sums here.  Hence rtol 1e-12 on losses and 1e-10 on per-tensor gradient norms."""
import copy
import os
import subprocess
import sys

import networkx as nx
import pytest
import torch

from nn_distributed_training_b200.models import FourierNet
from nn_distributed_training_b200.models.relu_nn import FFReLUNet

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F64 = torch.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _density_problem(backend, h1=256, B=1000, M=3000, N=3, loss="BCE", first="sin_relu", seed=0):
    from nn_distributed_training_b200.data.shards import Shard
    from nn_distributed_training_b200.problems import DistDensityProblem
    g = torch.Generator().manual_seed(seed)
    shards = []
    for i in range(N):
        x = ((torch.rand(M, 2, generator=g) - 0.5) * 1200).double()
        y = (torch.rand(M, generator=g) < 0.3).double()
        shards.append(Shard(x, y))
    val = Shard(((torch.rand(500, 2, generator=g) - 0.5) * 1200).double(), (torch.rand(500, generator=g) < 0.3).double())
    conf = {"problem_name": "d", "train_batch_size": B, "val_batch_size": 200,
            "metrics": ["forward_pass_count", "validation_loss", "consensus_error", "current_epoch"],
            "metrics_config": {"evaluate_frequency": 100}, "optimizer_config": {}}
    torch.manual_seed(seed)
    shape = [2, h1, 64, 64, 64, 1]
    base = FourierNet(shape, scale=0.05, dtype=F64) if first == "sin_relu" else FFReLUNet(shape, dtype=F64)
    lossf = {"BCE": torch.nn.BCELoss(), "MSE": torch.nn.MSELoss(), "L1": torch.nn.L1Loss()}[loss]
    return DistDensityProblem(nx.cycle_graph(N), base, lossf, shards, val, DEV, conf, backend=backend, seed=3)


def _pair(**kw):
    fused = _density_problem("fused", **kw)
    ref = _density_problem("torch", **kw)
    assert fused.backend == "fused" and ref.backend == "torch"
    assert fused.arena.dtype == ref.arena.dtype == F64
    ref.arena.theta.copy_(fused.arena.theta)
    return fused, ref


def _compare_steps(fused, ref, steps, first_layer_tol=1e-10):
    for step in range(steps):
        lf = fused.compute_grads().clone()
        lr = ref.compute_grads().clone()
        assert lf.dtype == F64
        torch.testing.assert_close(lf, lr, rtol=1e-12, atol=0)
        for s in fused.layout.slots:
            a = fused.arena.grad[:, s.offset: s.offset + s.numel]
            b = ref.arena.grad[:, s.offset: s.offset + s.numel]
            rel = ((a - b).norm() / b.norm().clamp_min(1e-300)).item()
            assert rel <= (first_layer_tol if s.name.startswith("seq.0") else 1e-10), (s.name, rel, step)
    assert (fused.calls == ref.calls).all()


@pytest.mark.parametrize("h1,B,M,loss,first", [
    (256, 1000, 3000, "BCE", "sin_relu"),
    (256, 77, 3000, "BCE", "sin_relu"),          # a batch smaller than one 64-row tile plus a ragged tile
    (64, 300, 3000, "MSE", "sin_relu"),
    (128, 1500, 3000, "L1", "sin_relu"),
    (256, 2048, 3000, "BCE", "sin_relu"),
    (128, 500, 3000, "MSE", "relu"),            # ReLU first layer (FFReLUNet: no output activation)
    (256, 300, 1000, "BCE", "sin_relu"),         # M % B != 0: step 4 draws the partial last batch of 100
])
def test_f64_train_kernel_matches_autograd(h1, B, M, loss, first, monkeypatch):
    monkeypatch.setenv("NNDT_FUSED_MLP", "0")    # the FFReLUNet reference runs nn.Sequential, not csrc/mlp_generic.cu
    fused, ref = _pair(h1=h1, B=B, M=M, loss=loss, first=first)
    _compare_steps(fused, ref, 5)


def test_f64_bce_saturation_matches_aten():
    """Logits spread over about +-40 for both labels: inside 27.6 < |z| < 37 ATen's 1e-12 clamp of p (1 - p) is active
    while p is not yet 0 or 1; beyond it log clamps at -100 and dL/dz is exactly 0 for the saturated side.

    The output-layer and hidden gradients keep the 1e-10 bound.  The first layer's are sums over rows whose dL/dz differ
    by many orders of magnitude and in sign (clamped band rows next to ordinary ones), and that cancellation costs about
    one more digit in either summation order (1.04e-10 measured on the bias of the first layer), hence 1e-9 there."""
    fused, ref = _pair(h1=256, B=1000, M=3000)
    with torch.no_grad():
        x = ref.shards.x.to(DEV, F64)
        z = torch.cat([ref.models[g].seq[:-1](x).reshape(-1) for g in range(3)])     # logits
        mu, a = z.mean(), 42.0 / (z - z.mean()).abs().max()
        for g in range(3):
            out = ref.models[g].seq[-2]
            out.weight.mul_(a)
            out.bias.sub_(mu).mul_(a)
        zs = torch.cat([ref.models[g].seq[:-1](x).reshape(-1) for g in range(3)])
    band = ((zs.abs() > 27.6) & (zs.abs() < 37)).sum().item()
    beyond = (zs.abs() >= 37).sum().item()
    assert band > 100 and beyond > 10 and zs.min() < -30 and zs.max() > 30, (band, beyond)
    fused.arena.theta.copy_(ref.arena.theta)
    _compare_steps(fused, ref, 3, first_layer_tol=1e-9)


def _online_problem(backend, tmp, opt_conf, B=700, metrics=None):
    import glob
    import numpy as np
    from nn_distributed_training_b200.floorplans.lidar import Lidar2D, OnlineTrajectoryLidarDataset, RandomPoseLidarDataset
    from nn_distributed_training_b200.floorplans.synthetic import write_dataset
    from nn_distributed_training_b200.problems import DistOnlineDensityProblem
    if not os.path.exists(os.path.join(tmp, "floor_img.png")):
        write_dataset(tmp, n_paths=3, seed=0)
    lidar = Lidar2D(os.path.join(tmp, "floor_img.png"), 8, 0.2, 10, 1.0, 20, 3, border_width=8)
    paths = sorted(glob.glob(os.path.join(tmp, "tight_paths", "*.npy")))
    np.random.seed(0)
    train = [OnlineTrajectoryLidarDataset(lidar, np.load(p), 4, 12, seed=5, node=i) for i, p in enumerate(paths)]
    val = RandomPoseLidarDataset(lidar, 10)
    conf = {"problem_name": "o", "train_batch_size": B, "val_batch_size": 300, "comm_radius": 300.0,
            "dynamic_graph": True, "save_models": False,
            "metrics": metrics or ["forward_pass_count", "train_loss_moving_average", "validation_loss", "consensus_error",
                                   "current_epoch"],
            "metrics_config": {"evaluate_frequency": 4, "tloss_decay": 0.2, "mesh_only_at_end": True},
            "optimizer_config": opt_conf}
    torch.manual_seed(0)
    base = FourierNet([2, 256, 64, 64, 64, 1], scale=0.05, dtype=F64)
    return DistOnlineDensityProblem(base, torch.nn.BCELoss(), train, val, DEV, conf, backend=backend, seed=5)


DSGD_C = {"alg_name": "dsgd", "alpha0": 0.001, "mu": 0.001, "outer_iterations": 10, "profile": False}
DSGT_C = {"alg_name": "dsgt", "alpha": 0.001, "init_grads": True, "outer_iterations": 10, "profile": False}
DINNO_C = {"alg_name": "dinno", "rho_init": 0.3, "rho_scaling": 1.0004, "outer_iterations": 10, "primal_iterations": 3,
           "primal_optimizer": "adam", "persistant_primal_opt": False, "primal_lr_start": 0.001,
           "primal_lr_finish": 0.0001, "lr_decay_type": "log", "profile": False}


def test_f64_online_window_sampler_matches_python(tmp_path):
    fused = _online_problem("fused", str(tmp_path), DSGD_C)
    ref = _online_problem("torch", str(tmp_path), DSGD_C)
    assert fused.backend == "fused"
    ref.arena.theta.copy_(fused.arena.theta)
    for step in range(12):          # windows hold 12 scans x 80 points = 960 draws: a switch every ~1.4 steps
        lf = fused.compute_grads().clone()
        lr = ref.compute_grads().clone()
        torch.testing.assert_close(lf, lr, rtol=1e-12, atol=0)
    assert (fused.positions() == ref.positions()).all()


def test_f64_eval_matches_torch(tmp_path):
    metrics = ["validation_loss", "mesh_grid_density"]
    fused = _online_problem("fused", str(tmp_path), DSGD_C, metrics=metrics)
    ref = _online_problem("torch", str(tmp_path), DSGD_C, metrics=metrics)
    ref.arena.theta.copy_(fused.arena.theta)
    vf, vr = fused._val_losses_local(), ref._val_losses_local()
    assert vf.dtype == F64
    torch.testing.assert_close(vf, vr, rtol=1e-12, atol=0)
    mf, mr = fused._mesh_all(), ref._mesh_all()
    assert mf.dtype == F64 and mf.shape == mr.shape
    torch.testing.assert_close(mf, mr, rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("name,conf", [("dinno", DINNO_C), ("dsgd", DSGD_C), ("dsgt", DSGT_C)])
def test_f64_fused_runs_track_torch_runs(tmp_path, name, conf):
    """Ten rounds, fused forward/backward + fused consensus kernels vs autograd + the torch consensus path.  Adam divides
    by sqrt(v): coordinates whose gradient is near zero can amplify the last-bit differences, so theta is compared by
    its relative norm."""
    from nn_distributed_training_b200.optimizers import DiNNO, DSGD, DSGT
    cls = {"dinno": DiNNO, "dsgd": DSGD, "dsgt": DSGT}[name]
    fused = _online_problem("fused", str(tmp_path), conf)
    ref = _online_problem("torch", str(tmp_path), conf)
    ref.arena.theta.copy_(fused.arena.theta)
    cls(fused, DEV, copy.deepcopy(conf)).train()
    cls(ref, DEV, dict(copy.deepcopy(conf), consensus_backend="torch")).train()
    assert len(fused.metrics["validation_loss"]) == len(ref.metrics["validation_loss"]) >= 3
    for key in ("validation_loss", "train_loss_moving_average"):
        for a, b in zip(fused.metrics[key], ref.metrics[key]):
            torch.testing.assert_close(a, b, rtol=1e-8, atol=0)
    assert fused.forward_cnt == ref.forward_cnt
    assert fused.metrics["forward_pass_count"] == ref.metrics["forward_pass_count"]
    rel = ((fused.arena.theta - ref.arena.theta).norm() / ref.arena.theta.norm()).item()
    assert rel <= 1e-8, rel


def test_f64_backend_selection(capsys):
    fused = _density_problem("auto")
    assert fused.backend == "fused" and fused.fused is not None and fused.fused.grad_part.dtype == F64
    assert "WARNING" not in capsys.readouterr().out
    from nn_distributed_training_b200.data.shards import Shard
    from nn_distributed_training_b200.problems import DistDensityProblem
    x = torch.rand(100, 2, dtype=F64)
    conf = {"problem_name": "d", "train_batch_size": 50, "val_batch_size": 50, "metrics": ["validation_loss"],
            "metrics_config": {"evaluate_frequency": 10}, "optimizer_config": {}}
    odd = DistDensityProblem(nx.cycle_graph(2), FourierNet([2, 100, 64, 64, 64, 1], 0.05, dtype=F64), torch.nn.BCELoss(),
                             [Shard(x, x[:, 0]), Shard(x, x[:, 1])], Shard(x, x[:, 0]), DEV, conf, backend="auto")
    assert odd.backend == "torch" and odd.fused is None
    assert "no fused forward/backward kernel" in capsys.readouterr().out


@pytest.mark.parametrize("name,conf", [("dinno", dict(DINNO_C, persistant_primal_opt=True, outer_iterations=6)),
                                       ("dsgt", dict(DSGT_C, outer_iterations=6))])
def test_f64_fused_runs_are_deterministic_and_resume_bit_exact(tmp_path, name, conf):
    """The kernel has no floating-point atomics: equal seeds give equal bits, and a checkpoint after an odd round resumed
    in a fresh problem ends where the uninterrupted run ends."""
    from nn_distributed_training_b200.optimizers import DiNNO, DSGT
    from nn_distributed_training_b200.parallel.context import DistContext
    from nn_distributed_training_b200.utils import checkpoint as ckpt
    cls = {"dinno": DiNNO, "dsgt": DSGT}[name]
    tmp = str(tmp_path)
    runs = []
    for _ in range(2):
        pr = _online_problem("fused", tmp, conf)
        cls(pr, DEV, copy.deepcopy(conf)).train()
        runs.append(pr)
    assert torch.equal(runs[0].arena.theta, runs[1].arena.theta)
    first = _online_problem("fused", tmp, conf)
    o1 = cls(first, DEV, copy.deepcopy(conf))
    ckpt.attach(o1, os.path.join(tmp, "ck"), "run", every=3, ctx=DistContext.single(torch.device(DEV)))
    o1.oits = 3
    o1.train()
    assert o1.k == 3
    second = _online_problem("fused", tmp, conf)
    o2 = cls(second, DEV, copy.deepcopy(conf))
    ckpt.attach(o2, os.path.join(tmp, "ck"), "run", every=3, ctx=DistContext.single(torch.device(DEV)), resume=True)
    assert o2.k == 3
    o2.train()
    assert torch.equal(second.arena.theta, runs[0].arena.theta)
    assert second.forward_cnt == runs[0].forward_cnt


def test_f64_online_runner_two_gpus_matches_single_process(tmp_path):
    """dist_online_dense_ex.py at experiment.dtype float64 under torchrun on two GPUs writes the results of the
    single-process run."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import glob

    import yaml
    from nn_distributed_training_b200.floorplans.synthetic import write_dataset
    floor = str(tmp_path / "floor")
    write_dataset(floor, n_paths=4, seed=0)
    with open(os.path.join(ROOT, "experiments", "dist_online_dense_PAPER_f64.yaml")) as f:
        base = yaml.safe_load(f)
    runner = os.path.join(ROOT, "experiments", "dist_online_dense_ex.py")
    outs = []
    for tag, nproc in (("single", 1), ("dist", 2)):
        conf = yaml.safe_load(yaml.safe_dump(base))
        e = conf["experiment"]
        out = str(tmp_path / tag)
        os.makedirs(out)
        e.update(output_metadir=out)
        e["data"].update(data_dir=floor, num_beams=8, beam_samps=10, collision_samps=20, spline_res=4,
                         num_validation_scans=20, border_width=8, num_scans_in_window=10, num_nodes=4)
        e["individual_training"].update(train_solo=False)
        for pc in conf["problem_configs"].values():
            pc.update(train_batch_size=300, val_batch_size=400, comm_radius=300.0, save_models=False)
            pc["metrics"] = [m for m in pc["metrics"] if m != "mesh_grid_density"]
            pc["metrics_config"].update(evaluate_frequency=3)
            pc["optimizer_config"]["outer_iterations"] = 5
        cfg = os.path.join(out, "o.yaml")
        with open(cfg, "w") as f:
            yaml.safe_dump(conf, f)
        if nproc == 1:
            cmd = [sys.executable, runner, cfg]
        else:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                   "--master-addr", "127.0.0.1", "--master-port", "29631", runner, cfg]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS="2"),
                           cwd=os.path.join(ROOT, "experiments"))
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        assert "no fused forward/backward kernel" not in r.stdout
        outs.append(glob.glob(os.path.join(out, "*_dist_online_dense_PAPER_f64"))[0])
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(outs[0], "*_results.pt")))
    assert names and names == sorted(os.path.basename(p) for p in glob.glob(os.path.join(outs[1], "*_results.pt")))
    for n in names:
        a = torch.load(os.path.join(outs[0], n), weights_only=False)
        b = torch.load(os.path.join(outs[1], n), weights_only=False)
        va, vb = torch.stack(a["validation_loss"]), torch.stack(b["validation_loss"])
        assert va.dtype == F64 and va.shape == vb.shape and va.shape[1] == 4
        torch.testing.assert_close(va, vb, rtol=1e-10, atol=0)
        assert a["forward_pass_count"] == b["forward_pass_count"]
