"""Property tests of topology, sampling and the consensus updates (SURVEY §4 item 4)."""
import copy
import os

import networkx as nx
import numpy as np
import pytest
import torch

from nn_distributed_training_b200.data.sampler import (BatchSchedule, OnlineWindowSchedule, feistel_permute, mix_key)
from nn_distributed_training_b200.models import FFReLUNet, FourierNet, MNISTConvNet
from nn_distributed_training_b200.optimizers import DiNNO, DSGD, DSGT
from nn_distributed_training_b200.parallel.arena import FlatLayout
from nn_distributed_training_b200.problems import DistMNISTProblem
from nn_distributed_training_b200.utils import checkpoint as ckpt
from nn_distributed_training_b200.utils import graph_generation as gg


@pytest.mark.parametrize("graph", [nx.cycle_graph(7), nx.wheel_graph(6), nx.complete_graph(5), nx.path_graph(4),
                                   nx.erdos_renyi_graph(9, 0.5, seed=2)])
def test_metropolis_is_symmetric_doubly_stochastic(graph):
    W = gg.get_metropolis(graph, dtype=torch.float64)
    assert torch.allclose(W, W.T)
    assert torch.allclose(W.sum(0), torch.ones(len(graph), dtype=torch.float64))
    assert torch.allclose(W.sum(1), torch.ones(len(graph), dtype=torch.float64))
    assert (W >= 0).all()
    A = torch.as_tensor(nx.to_numpy_array(graph)) > 0
    assert ((W > 0) & ~torch.eye(len(graph), dtype=torch.bool) == A).all()


def metropolis_graphs():
    return [nx.cycle_graph(10), nx.wheel_graph(7), nx.erdos_renyi_graph(12, 0.4, seed=1)]


@pytest.fixture(scope="module")
def golden():
    """The reference's own outputs on the inputs built here (written by oracle/make_golden.py)."""
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_properties.npz")) as z:
        return dict(z)


def test_metropolis_matches_reference(golden):
    for i, g in enumerate(metropolis_graphs()):
        torch.testing.assert_close(gg.get_metropolis(g, dtype=torch.float64), torch.as_tensor(golden[f"metropolis/{i}"]))


def test_complete_graph_metropolis_is_uniform():
    assert torch.allclose(gg.get_metropolis(nx.complete_graph(8)), torch.full((8, 8), 0.125))


def test_generate_from_conf_types_and_errors():
    for kind in ("wheel", "cycle", "complete", "path", "star"):
        N, g = gg.generate_from_conf({"num_nodes": 6, "type": kind})
        assert N == 6 and g.number_of_nodes() == 6 and nx.is_connected(g)
    N, g = gg.generate_from_conf({"num_nodes": 8, "type": "random", "p": 0.5, "gen_attempts": 50})
    assert nx.is_connected(g)
    with pytest.raises(NameError):
        gg.generate_from_conf({"num_nodes": 30, "type": "random", "p": 0.0, "gen_attempts": 2})
    with pytest.raises(NameError):
        gg.generate_from_conf({"num_nodes": 3, "type": "hypercube"})


def test_disk_graphs():
    import random
    g = gg.disk_with_fied(12, 1.0, rng=random.Random(0))
    fied = gg.fiedler_value(gg.adjacency(g))
    assert abs(fied - 1.0) < 0.011 and nx.is_connected(g)
    poses = np.array([[0, 0], [1, 0], [5, 5]], dtype=float)
    g2, conn = gg.euclidean_disk_graph(poses, 1.5)
    assert set(g2.edges()) == {(0, 1)} and not conn
    g3, conn3 = gg.euclidean_disk_graph(poses, 10.0)
    assert conn3 and g3.number_of_edges() == 3
    assert gg.gen_delaunay(10).number_of_nodes() == 10


def test_feistel_is_a_bijection_and_keyed():
    for m in (1, 2, 3, 17, 64, 100, 1000, 4097):
        p = feistel_permute(torch.arange(m), m, mix_key(3, 1, 0))
        assert sorted(p.tolist()) == list(range(m))
    a = feistel_permute(torch.arange(500), 500, mix_key(3, 1, 0))
    b = feistel_permute(torch.arange(500), 500, mix_key(3, 1, 1))
    assert (a != b).float().mean() > 0.9


def test_batch_schedule_matches_dataloader_structure():
    ds = torch.utils.data.TensorDataset(torch.arange(150))
    dl = torch.utils.data.DataLoader(ds, batch_size=64, shuffle=True)
    sizes = [len(b[0]) for b in dl]
    s = BatchSchedule(150, 64)
    assert [s.locate(c)[2] for c in range(3)] == sizes
    seen = torch.cat([s.indices(c, 0, 0) for c in range(3)])
    assert sorted(seen.tolist()) == list(range(150))               # one epoch visits every sample once
    assert [s.epochs_completed(c) for c in (0, 3, 4, 6, 7)] == [0, 0, 1, 1, 2]


def test_online_window_schedule_matches_reference_logic():
    """Replay the reference's gen_next_index_list state machine (lidar.py:397-424)."""
    for T, Wn, S in [(10, 3, 5), (11, 3, 4), (7, 7, 2), (9, 2, 3)]:
        cur, wins = 0, []
        for _ in range(12):
            if cur + Wn >= T:
                if cur == T - 1:
                    cur = Wn
                    lb, ub = S * (cur - Wn), S * cur
                else:
                    lb, ub = S * cur, S * T
                    cur = T - 1
            else:
                cur += Wn
                lb, ub = S * (cur - Wn), S * cur
            wins.append((lb, ub, cur))
        sch = OnlineWindowSchedule(T, S, Wn)
        assert [sch.window(w) for w in range(12)] == wins
        n0 = wins[0][1] - wins[0][0]
        idx = sch.indices(0, n0, 0, 0)
        assert sorted(idx.tolist()) == list(range(wins[0][0], wins[0][1]))
        assert sch.scan_cursor_at(0) == wins[0][2] and sch.scan_cursor_at(n0) == wins[0][2]
        assert sch.scan_cursor_at(n0 + 1) == wins[1][2]


def test_flat_layout_alignment_and_roundtrip():
    for m in (MNISTConvNet(3, 5, 64), FourierNet([2, 256, 64, 64, 64, 1], 0.05), FFReLUNet([12, 64, 64, 5])):
        lay = FlatLayout.from_module(m)
        assert lay.n == sum(p.numel() for p in m.parameters())
        assert all(s.offset % 4 == 0 for s in lay.slots) and lay.n_pad % 128 == 0
        row = torch.zeros(lay.n_pad)
        lay.flatten(m, row)
        assert torch.equal(lay.compact(row), torch.nn.utils.parameters_to_vector(m.parameters()).detach())
    assert MNISTConvNet(3, 5, 64).spec.fc1_in == 432
    assert sum(p.numel() for p in MNISTConvNet(3, 5, 64).parameters()) == 28440
    assert sum(p.numel() for p in FourierNet([2, 256, 64, 64, 64, 1], 0.05).parameters()) == 25601


def _mnist_problem(N, graph, conf, seed=0):
    g = torch.Generator().manual_seed(seed)
    train = [torch.utils.data.TensorDataset(torch.randn(40, 1, 28, 28, generator=g), torch.randint(0, 10, (40,), generator=g))
             for _ in range(N)]
    val = torch.utils.data.TensorDataset(torch.randn(30, 1, 28, 28, generator=g), torch.randint(0, 10, (30,), generator=g))
    pconf = {"problem_name": "p", "train_batch_size": 16, "val_batch_size": 16,
             "metrics": ["forward_pass_count", "validation_loss", "consensus_error", "top1_accuracy", "current_epoch"],
             "metrics_config": {"evaluate_frequency": 100}, "optimizer_config": conf}
    torch.manual_seed(seed)
    pr = DistMNISTProblem(graph, MNISTConvNet(3, 5, 64), torch.nn.NLLLoss(), train, val, "cpu", pconf)
    # break the symmetric start so the invariants are non-trivial
    pr.arena.theta.add_(0.05 * torch.randn(pr.arena.theta.shape, generator=g) * (pr.arena.theta != 0))
    return pr


def test_dsgd_jacobi_mean_evolves_by_mean_gradient():
    """theta+ = W theta - alpha g with doubly stochastic W  =>  mean(theta+) = mean(theta) - alpha mean(g)."""
    conf = {"alg_name": "dsgd", "alpha0": 0.05, "mu": 0.0, "outer_iterations": 1, "profile": False}
    pr = _mnist_problem(5, nx.wheel_graph(5), conf)
    before = pr.arena.theta.mean(0).clone()
    DSGD(pr, "cpu", conf).train()
    torch.testing.assert_close(pr.arena.theta.mean(0), before - 0.05 * pr.arena.grad.mean(0), rtol=1e-4, atol=1e-6)


def test_dsgt_tracker_sum_equals_gradient_sum():
    conf = {"alg_name": "dsgt", "alpha": 0.02, "init_grads": True, "outer_iterations": 4, "profile": False}
    pr = _mnist_problem(6, nx.cycle_graph(6), conf)
    opt = DSGT(pr, "cpu", conf)
    opt.train()
    torch.testing.assert_close(opt.y.sum(0), opt.g.sum(0), rtol=1e-4, atol=1e-5)


def test_dinno_duals_sum_to_zero_on_undirected_graph():
    conf = {"alg_name": "dinno", "rho_init": 0.5, "rho_scaling": 1.01, "outer_iterations": 3, "primal_iterations": 2,
            "primal_optimizer": "adam", "persistant_primal_opt": False, "primal_lr_start": 0.005,
            "primal_lr_finish": 0.0005, "lr_decay_type": "log", "profile": False}
    pr = _mnist_problem(5, nx.erdos_renyi_graph(5, 0.7, seed=1), conf)
    opt = DiNNO(pr, "cpu", conf)
    opt.train()
    assert opt.duals.abs().max() > 1e-4
    assert opt.duals.sum(0).abs().max() < 1e-4 * opt.duals.abs().max() * 10


def test_isolated_node_takes_a_local_step():
    """A node with no neighbors (disconnected graph) must not crash DiNNO (SURVEY Q19)."""
    g = nx.Graph()
    g.add_nodes_from(range(3))
    g.add_edge(0, 1)
    conf = {"alg_name": "dinno", "rho_init": 0.5, "rho_scaling": 1.0, "outer_iterations": 2, "primal_iterations": 1,
            "primal_optimizer": "sgd", "persistant_primal_opt": False, "primal_lr_start": 0.01,
            "primal_lr_finish": 0.01, "lr_decay_type": "constant", "profile": False}
    pr = _mnist_problem(3, g, conf)
    t0 = pr.arena.theta.clone()
    opt = DiNNO(pr, "cpu", conf)
    opt.train()
    assert torch.isfinite(pr.arena.theta).all() and not torch.equal(pr.arena.theta[2], t0[2])
    assert opt.duals[2].abs().max() == 0


@pytest.mark.parametrize("alg", ["dinno", "dsgd", "dsgt"])
def test_checkpoint_resume_is_bit_exact(tmp_path, alg):
    from nn_distributed_training_b200.parallel.context import DistContext
    confs = {
        "dinno": {"alg_name": "dinno", "rho_init": 0.5, "rho_scaling": 1.01, "outer_iterations": 6, "primal_iterations": 2,
                  "primal_optimizer": "adam", "persistant_primal_opt": True, "primal_lr_start": 0.005,
                  "primal_lr_finish": 0.0005, "lr_decay_type": "log", "profile": False},
        "dsgd": {"alg_name": "dsgd", "alpha0": 0.05, "mu": 0.01, "outer_iterations": 6, "profile": False},
        "dsgt": {"alg_name": "dsgt", "alpha": 0.02, "init_grads": True, "outer_iterations": 6, "profile": False},
    }
    conf = confs[alg]
    cls = {"dinno": DiNNO, "dsgd": DSGD, "dsgt": DSGT}[alg]
    full = _mnist_problem(4, nx.cycle_graph(4), conf)
    cls(full, "cpu", conf).train()

    first = _mnist_problem(4, nx.cycle_graph(4), conf)
    o1 = cls(first, "cpu", conf)
    cp = ckpt.attach(o1, str(tmp_path), "run", every=3, ctx=DistContext.single())
    o1.oits = 3                      # "crash" after round 3
    o1.train()
    assert o1.k == 3
    second = _mnist_problem(4, nx.cycle_graph(4), conf)
    o2 = cls(second, "cpu", conf)
    ckpt.attach(o2, str(tmp_path), "run", every=3, ctx=DistContext.single(), resume=True)
    assert o2.k == 3
    o2.train()
    assert torch.equal(second.arena.theta, full.arena.theta)
    assert second.forward_cnt == full.forward_cnt


def test_link_drop_fault_injection_changes_graph_and_training_survives():
    conf = {"alg_name": "dinno", "rho_init": 0.5, "rho_scaling": 1.0, "outer_iterations": 5, "primal_iterations": 1,
            "primal_optimizer": "sgd", "persistant_primal_opt": False, "primal_lr_start": 0.01,
            "primal_lr_finish": 0.01, "lr_decay_type": "constant", "profile": False}
    pr = _mnist_problem(5, nx.cycle_graph(5), conf)
    pr.conf["fault_injection"] = {"link_drop_prob": 0.5, "seed": 3, "from_round": 1, "to_round": 4}
    pr._init_faults()
    plan = pr.plan_graphs(5, 0, 1)
    assert plan[0].number_of_edges() == 5 and plan[4].number_of_edges() == 5
    assert any(g.number_of_edges() < 5 for g in plan[1:4])
    DiNNO(pr, "cpu", conf).train()
    assert torch.isfinite(pr.arena.theta).all()
    # the eager path walked the same graph sequence as the plan
    assert pr._graph_round == 5


def lidar_inputs():
    """The reference's floor plan and first tight path (shipped unchanged under floorplans/32_data)."""
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "floorplans", "32_data")
    return os.path.join(d, "floor_img.png"), np.load(os.path.join(d, "tight_paths", "1.npy"))


def lidar_trajectory(interpolate_waypoints, wp, lidar):
    return interpolate_waypoints(wp[:, 0], wp[:, 1], 1)[::6] * np.array([lidar.nx * 0.5, lidar.ny * 0.5])


def test_lidar_matches_reference_scans(golden):
    """Vectorised lidar vs the reference's per-beam Python loops on the reference's own floor plan."""
    from nn_distributed_training_b200.floorplans.lidar import ClippedLidar2D, Lidar2D, interpolate_waypoints
    img, wp = lidar_inputs()
    mine = Lidar2D(img, 12, 0.2, 15, 1.0, 30, 3, border_width=30)
    np.testing.assert_allclose(interpolate_waypoints(wp[:, 0], wp[:, 1], 3), golden["lidar/interp3"])
    traj = lidar_trajectory(interpolate_waypoints, wp, mine)
    np.testing.assert_allclose(mine.scan_batch(traj), golden["lidar/scans"], rtol=1e-9, atol=1e-9)
    cm = ClippedLidar2D(img, 12, 0.2, 15, border_width=30)
    for i, p in enumerate(traj[:4]):
        np.testing.assert_allclose(cm.scan(p.reshape(1, 2)), golden[f"lidar/clipped/{i}"], rtol=1e-9, atol=1e-9)


def test_round_timer_as_profiler_hook():
    from nn_distributed_training_b200.utils.timing import RoundTimer
    conf = {"alg_name": "dsgd", "alpha0": 0.05, "mu": 0.0, "outer_iterations": 6, "profile": False}
    pr = _mnist_problem(3, nx.cycle_graph(3), conf)
    t = RoundTimer(warmup=2)
    DSGD(pr, "cpu", conf).train(profiler=t)
    assert t.ms_per_round() is not None and t.ms_per_round() > 0


def test_choose_spb_fills_one_wave():
    """Samples per training CTA: smallest value whose L x ceil(B / spb) CTAs fit in one wave of the SMs."""
    from nn_distributed_training_b200.ops.mnist_fused import SPB, choose_spb
    assert choose_spb(64, 10, 148) == 5          # bench configuration: 13 slices x 10 nodes = 130 CTAs
    assert choose_spb(64, 1, 148) == 4
    assert choose_spb(64, 18, 148) == 8          # 8 x 18 = 144
    assert choose_spb(64, 40, 148) == SPB        # nothing fits: fewest CTAs
    for B in (16, 32, 64, 100):
        for L in (1, 3, 10, 18, 30):
            spb = choose_spb(B, L, 148)
            assert 4 <= spb <= SPB
            if spb > 4:                          # a smaller value would not have fitted
                assert L * -(-B // (spb - 1)) > 148


def test_numa_binding_helper_is_safe_without_nvml(monkeypatch):
    """parallel/context.py: bind_to_local_cpus never raises and only ever narrows the affinity to NVML's local CPUs."""
    import os
    from nn_distributed_training_b200.parallel import context as C
    assert C.cpus_from_mask([0b1011, 0b1]) == {0, 1, 3, 64}
    before = os.sched_getaffinity(0)
    monkeypatch.setenv("NNDT_NUMA_BIND", "0")
    assert C.bind_to_local_cpus(0) is None

    class FakeNvml:            # a GPU whose local CPUs are the first half of the allowed set
        def __init__(self, cpus): self.cpus = cpus
        def nvmlDeviceGetHandleByUUID(self, u): raise RuntimeError("no uuid")
        def nvmlDeviceGetHandleByIndex(self, i): return i
        def nvmlDeviceGetCpuAffinity(self, h, n):
            words = [0] * n
            for c in self.cpus:
                words[c // 64] |= 1 << (c % 64)
            return words

    monkeypatch.setenv("NNDT_NUMA_BIND", "1")
    allowed = sorted(before)
    half = set(allowed[: max(1, len(allowed) // 2)])
    got = C.bind_to_local_cpus(0, min_cpus=1, nvml=FakeNvml(half))
    try:
        if len(allowed) >= 2:
            assert got == half and os.sched_getaffinity(0) == half
        else:
            assert got is None
        # a mask that would leave too few CPUs is ignored
        os.sched_setaffinity(0, before)
        assert C.bind_to_local_cpus(0, min_cpus=len(allowed) + 1, nvml=FakeNvml(half)) is None
        assert os.sched_getaffinity(0) == before
    finally:
        os.sched_setaffinity(0, before)
